// factorize.cu -- GP factorisations on the device (fp64):
//   pilco_gp_factorize    MGPR.calculate_factorizations   pilco/models/mgpr.py:81-89  (gp0.m:46-61)
//   pilco_fitc_factorize  SMGPR.calculate_factorizations  pilco/models/smgpr.py:24-45 (gp1.m:52-82)
// Building blocks: SE-ARD (cross-)Gram kernel, blocked right-looking Cholesky (one CTA per matrix),
// blocked triangular inverse, a batched fp64 GEMM with transposes, blocked triangular solves for beta.
// These run once per set_data / hyper-parameter change (dynamics GP) or once per loss evaluation
// (RBF policy, bf<=128), never inside the H-step loop.
#include "common.cuh"

#define FB 32                     // factorisation block size

// -------------------------------------------------------------------------------------------------
// SE-ARD Gram:  K[i][j] = sf2 exp(-0.5 sum_d ((x1_i - x2_j)/ell_d)^2) + diag_add*(i==j)
// grid (ceil(n2/32), ceil(n1/8), batch) block (32, 8).  Output leading dimension ldo; entries with
// i>=n1 or j>=n2 inside [0,rows_out) x [0,cols_out) are written as 0 (1 on the diagonal if unit_pad).
// -------------------------------------------------------------------------------------------------
struct GramArgs {
    int n1, n2, D, E;
    const double* X1; long long X1_bs;       // [n1,D] per batch b
    const double* X2; long long X2_bs;       // [n2,D]
    const double* ell; long long ell_bs;     // [E,D]
    const double* sf2; long long sf2_bs;     // [E]
    const double* dadd; long long dadd_bs;   // [E] added on the diagonal (or NULL)
    double dconst;                           // constant added on the diagonal
    double* out; int ldo; long long out_ms;  // matrix stride (per (b,e))
    int rows_out, cols_out, unit_pad;
};

__global__ void __launch_bounds__(256) gram_kernel(GramArgs g) {
    PDL_ENTRY();
    const int z = blockIdx.z, bidx = z / g.E, e = z % g.E;
    const int j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= g.rows_out || j >= g.cols_out) return;
    double* out = g.out + (size_t)z * g.out_ms;
    double v;
    if (i < g.n1 && j < g.n2) {
        const double* x1 = g.X1 + (size_t)bidx * g.X1_bs + (size_t)i * g.D;
        const double* x2 = g.X2 + (size_t)bidx * g.X2_bs + (size_t)j * g.D;
        const double* ell = g.ell + (size_t)bidx * g.ell_bs + (size_t)e * g.D;
        double d2 = 0.0;
        for (int d = 0; d < g.D; ++d) { const double t = (x1[d] - x2[d]) / ell[d]; d2 = fma(t, t, d2); }
        v = g.sf2[(size_t)bidx * g.sf2_bs + e] * exp(-0.5 * d2);
        if (i == j) v += g.dconst + (g.dadd ? g.dadd[(size_t)bidx * g.dadd_bs + e] : 0.0);
    } else {
        v = (g.unit_pad && i == j) ? 1.0 : 0.0;
    }
    out[(size_t)i * g.ldo + j] = v;
}

// -------------------------------------------------------------------------------------------------
// Blocked right-looking Cholesky, in place, lower triangle, one CTA (256 threads) per matrix.
// Only the lower triangle is meaningful on exit.  info[b] |= 2 if a pivot is not positive.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) chol_kernel(int n, double* Aall, int ld, long long ms, int mats_per_b, int* info) {
    PDL_ENTRY();
    __shared__ double sD[FB][FB + 1];
    __shared__ double sPi[64][FB + 1];
    __shared__ double sPj[64][FB + 1];
    __shared__ int sfail;
    double* A = Aall + (size_t)blockIdx.x * ms;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) sfail = 0;
    for (int k0 = 0; k0 < n; k0 += FB) {
        const int kb = min(FB, n - k0);
        __syncthreads();
        for (int e = tid; e < FB * FB; e += 256) {
            const int i = e / FB, j = e % FB;
            sD[i][j] = (i < kb && j < kb) ? A[(size_t)(k0 + i) * ld + k0 + j] : (i == j ? 1.0 : 0.0);
        }
        __syncthreads();
        if (warp == 0) {                                   // left-looking Cholesky of the diagonal block, lane = row
            for (int j = 0; j < kb; ++j) {
                double v = sD[lane][j];
                for (int k = 0; k < j; ++k) v = fma(-sD[lane][k], sD[j][k], v);
                double piv = __shfl_sync(0xffffffffu, v, j);
                if (!(piv > 0.0)) { if (lane == 0) sfail = 1; piv = 1.0; }
                const double rp = 1.0 / sqrt(piv);
                __syncwarp();
                if (lane >= j) sD[lane][j] = (lane == j) ? sqrt(piv) : v * rp;
                __syncwarp();
            }
        }
        __syncthreads();
        for (int e = tid; e < kb * kb; e += 256) {          // write the factored block back
            const int i = e / kb, j = e % kb;
            A[(size_t)(k0 + i) * ld + k0 + j] = (j <= i) ? sD[i][j] : 0.0;
        }
        // panel: rows below the block, one thread per row:  x L_kk^T = a
        for (int i = k0 + kb + tid; i < n; i += 256) {
            double x[FB];
            double* arow = A + (size_t)i * ld + k0;
#pragma unroll
            for (int j = 0; j < FB; ++j) x[j] = j < kb ? arow[j] : 0.0;
#pragma unroll
            for (int j = 0; j < FB; ++j) {
                if (j < kb) {
                    double v = x[j];
#pragma unroll
                    for (int k = 0; k < j; ++k) v = fma(-x[k], sD[j][k], v);
                    x[j] = v / sD[j][j];
                }
            }
#pragma unroll
            for (int j = 0; j < FB; ++j) if (j < kb) arow[j] = x[j];
        }
        __syncthreads();
        // trailing update A[i][j] -= sum_k L[i][k0+k] L[j][k0+k], lower triangle, 64x64 tiles
        const int t0 = k0 + kb;
        if (t0 >= n) break;
        const int ntile = (n - t0 + 63) / 64;
        const int ty = tid / 16, tx = tid % 16;
        for (int ti = 0; ti < ntile; ++ti) {
            for (int tj = 0; tj <= ti; ++tj) {
                __syncthreads();
                for (int e = tid; e < 64 * FB; e += 256) {
                    const int rr = e / FB, k = e % FB;
                    const int gi = t0 + ti * 64 + rr, gj = t0 + tj * 64 + rr;
                    sPi[rr][k] = (gi < n && k < kb) ? A[(size_t)gi * ld + k0 + k] : 0.0;
                    sPj[rr][k] = (gj < n && k < kb) ? A[(size_t)gj * ld + k0 + k] : 0.0;
                }
                __syncthreads();
                double acc[4][4];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
                for (int k = 0; k < FB; ++k) {
                    double pi[4], pj[4];
#pragma unroll
                    for (int a = 0; a < 4; ++a) { pi[a] = sPi[ty + 16 * a][k]; pj[a] = sPj[tx + 16 * a][k]; }
#pragma unroll
                    for (int a = 0; a < 4; ++a)
#pragma unroll
                        for (int b = 0; b < 4; ++b) acc[a][b] = fma(pi[a], pj[b], acc[a][b]);
                }
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const int gi = t0 + ti * 64 + ty + 16 * a, gj = t0 + tj * 64 + tx + 16 * b;
                        if (gi < n && gj <= gi) A[(size_t)gi * ld + gj] -= acc[a][b];
                    }
            }
        }
    }
    __syncthreads();
    if (tid == 0 && sfail && info) atomicOr(&info[blockIdx.x / mats_per_b], 2);
}

// -------------------------------------------------------------------------------------------------
// inverse of the FB x FB diagonal blocks of a lower-triangular L:  X[I][I] = L[I][I]^-1
// grid (nblocks, batch), one warp; lane = column.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(32) tri_diag_inv_kernel(int n, const double* Lall, int ld, long long ms,
                                                          double* Xall, int ldx, long long xs) {
    __shared__ double sL[FB][FB + 1];
    __shared__ double sX[FB][FB + 1];
    const int I = blockIdx.x, lane = threadIdx.x;
    const double* L = Lall + (size_t)blockIdx.y * ms;
    double* X = Xall + (size_t)blockIdx.y * xs;
    const int k0 = I * FB, kb = min(FB, n - k0);
    for (int i = 0; i < FB; ++i)
        sL[i][lane] = (i < kb && lane < kb) ? L[(size_t)(k0 + i) * ld + k0 + lane] : (i == lane ? 1.0 : 0.0);
    __syncwarp();
    const int c = lane;
    for (int i = 0; i < FB; ++i) {
        double v = (i == c) ? 1.0 : 0.0;
        for (int k = c; k < i; ++k) v = fma(-sL[i][k], sX[k][c], v);
        sX[i][c] = (i >= c) ? v / sL[i][i] : 0.0;
    }
    __syncwarp();
    for (int i = 0; i < kb; ++i) if (lane < kb) X[(size_t)(k0 + i) * ldx + k0 + lane] = sX[i][lane];
}

// -------------------------------------------------------------------------------------------------
// batched GEMM  C = alpha op(A) op(B) + beta C   (row-major; op = transpose if flag set)
// grid (ceil(n/64), ceil(m/64), batch), 256 threads, 4x4 per thread, k-tile 16.
// -------------------------------------------------------------------------------------------------
struct GemmArgs {
    int m, n, k; int ta, tb;
    double alpha, beta;
    const double* A; int lda; long long sa;
    const double* B; int ldb; long long sb;
    double* C; int ldc; long long sc;
};

__global__ void __launch_bounds__(256) gemm_kernel(GemmArgs g) {
    __shared__ double sA[16][64 + 1];
    __shared__ double sB[16][64 + 1];
    const double* A = g.A + (size_t)blockIdx.z * g.sa;
    const double* B = g.B + (size_t)blockIdx.z * g.sb;
    double* C = g.C + (size_t)blockIdx.z * g.sc;
    const int tid = threadIdx.x, ty = tid / 16, tx = tid % 16;
    const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
    double acc[4][4];
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int k0 = 0; k0 < g.k; k0 += 16) {
        for (int e = tid; e < 16 * 64; e += 256) {
            int kk, ii;
            if (g.ta) { ii = e % 64; kk = e / 64; } else { kk = e % 16; ii = e / 16; }
            const int gi = i0 + ii, gk = k0 + kk;
            double v = 0.0;
            if (gi < g.m && gk < g.k) v = g.ta ? A[(size_t)gk * g.lda + gi] : A[(size_t)gi * g.lda + gk];
            sA[kk][ii] = v;
        }
        for (int e = tid; e < 16 * 64; e += 256) {
            int kk, jj;
            if (g.tb) { kk = e % 16; jj = e / 16; } else { jj = e % 64; kk = e / 64; }
            const int gj = j0 + jj, gk = k0 + kk;
            double v = 0.0;
            if (gj < g.n && gk < g.k) v = g.tb ? B[(size_t)gj * g.ldb + gk] : B[(size_t)gk * g.ldb + gj];
            sB[kk][jj] = v;
        }
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < 16; ++kk) {
            double a[4], b[4];
#pragma unroll
            for (int x = 0; x < 4; ++x) { a[x] = sA[kk][ty + 16 * x]; b[x] = sB[kk][tx + 16 * x]; }
#pragma unroll
            for (int x = 0; x < 4; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) acc[x][y] = fma(a[x], b[y], acc[x][y]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int x = 0; x < 4; ++x)
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const int gi = i0 + ty + 16 * x, gj = j0 + tx + 16 * y;
            if (gi < g.m && gj < g.n) {
                double* c = C + (size_t)gi * g.ldc + gj;
                *c = g.alpha * acc[x][y] + (g.beta != 0.0 ? g.beta * (*c) : 0.0);
            }
        }
}

// fp64 tensor-core variant (round 2): same contract, CTA tile 64 x 64, K tile 16, 8 warps as 4 (m) x 2 (n), warp tile
// 16 x 32 = 2 x 4 DMMA.8x8x4 accumulators.  Operand tiles staged K-major in shared memory with row stride 68
// (= 4 mod 16: the DMMA fragment reads of a half-warp hit 16 distinct bank pairs).  Used for every product of the
// factorisations and training objectives (iK = L^-T L^-1, FITC V V', B = V diag(1/nu) V', block-inverse updates ...).
#define GD_LD 68
__global__ void __launch_bounds__(256) gemm_dmma_kernel(GemmArgs g) {
    PDL_ENTRY();
    __shared__ double sA[16][GD_LD];
    __shared__ double sB[16][GD_LD];
    const double* A = g.A + (size_t)blockIdx.z * g.sa;
    const double* B = g.B + (size_t)blockIdx.z * g.sb;
    double* C = g.C + (size_t)blockIdx.z * g.sc;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int gq = lane >> 2, t = lane & 3;
    const int wm = (warp >> 1) * 16, wn = (warp & 1) * 32;      // warp tile origin inside the CTA tile
    const int i0 = blockIdx.y * 64, j0 = blockIdx.x * 64;
    double acc[2][4][2];
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b][0] = acc[a][b][1] = 0.0;
    for (int k0 = 0; k0 < g.k; k0 += 16) {
        for (int e = tid; e < 16 * 64; e += 256) {
            int kk, ii;
            if (g.ta) { ii = e % 64; kk = e / 64; } else { kk = e % 16; ii = e / 16; }
            const int gi = i0 + ii, gk = k0 + kk;
            double v = 0.0;
            if (gi < g.m && gk < g.k) v = g.ta ? A[(size_t)gk * g.lda + gi] : A[(size_t)gi * g.lda + gk];
            sA[kk][ii] = v;
        }
        for (int e = tid; e < 16 * 64; e += 256) {
            int kk, jj;
            if (g.tb) { kk = e % 16; jj = e / 16; } else { jj = e % 64; kk = e / 64; }
            const int gj = j0 + jj, gk = k0 + kk;
            double v = 0.0;
            if (gj < g.n && gk < g.k) v = g.tb ? B[(size_t)gj * g.ldb + gk] : B[(size_t)gk * g.ldb + gj];
            sB[kk][jj] = v;
        }
        __syncthreads();
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
            double af[2], bf[4];
#pragma unroll
            for (int a = 0; a < 2; ++a) af[a] = sA[4 * ks + t][wm + 8 * a + gq];     // A[m = row gq][k = t]
#pragma unroll
            for (int b = 0; b < 4; ++b) bf[b] = sB[4 * ks + t][wn + 8 * b + gq];     // B[k = t][n = col gq]
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 4; ++b) dmma884(acc[a][b][0], acc[a][b][1], af[a], bf[b]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b)
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int gi = i0 + wm + 8 * a + gq, gj = j0 + wn + 8 * b + 2 * t + c;     // C[row gq][cols 2t, 2t+1]
                if (gi < g.m && gj < g.n) {
                    double* cp = C + (size_t)gi * g.ldc + gj;
                    *cp = g.alpha * acc[a][b][c] + (g.beta != 0.0 ? g.beta * (*cp) : 0.0);
                }
            }
}

static int gemm(cudaStream_t st, int batch, int m, int n, int k, int ta, int tb, double alpha,
                const double* A, int lda, long long sa, const double* B, int ldb, long long sb,
                double beta, double* C, int ldc, long long sc) {
    if (m <= 0 || n <= 0) return PILCO_OK;
    GemmArgs g{m, n, k, ta, tb, alpha, beta, A, lda, sa, B, ldb, sb, C, ldc, sc};
    dim3 grid((n + 63) / 64, (m + 63) / 64, batch);
    static int use_dmma = -1;                                   // PILCO_GEMM_DFMA=1: the round-1 DFMA kernel (A/B switch)
    if (use_dmma < 0) { const char* e = getenv("PILCO_GEMM_DFMA"); use_dmma = (e && e[0] == '1') ? 0 : 1; }
    if (use_dmma) launch_pri(pilco_small_grid(grid), gemm_dmma_kernel, grid, dim3(256), 0, st, g);
    else gemm_kernel<<<grid, 256, 0, st>>>(g);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

// -------------------------------------------------------------------------------------------------
// Cholesky at scale (round 2): for n >= CHOL_MULTI_N the right-looking blocked algorithm runs ACROSS CTAs -- per block
// column: diagonal block (one CTA per matrix), panel solve (one thread per row, 256 rows per CTA), trailing update
// A22 -= L21 L21' as ONE batched DMMA GEMM over the whole remaining square (the upper half is redundant work, but it
// is tensor-core work spread over the machine instead of 64 x 64 DFMA tiles on the single CTA of chol_kernel).
// -------------------------------------------------------------------------------------------------
#define CHOL_MULTI_N 512
__global__ void __launch_bounds__(32) chol_diag_kernel(int n, int k0, double* Aall, int ld, long long ms, int mats_per_b, int* info) {
    PDL_ENTRY();
    __shared__ double sD[FB][FB + 1];
    double* A = Aall + (size_t)blockIdx.x * ms;
    const int lane = threadIdx.x, kb = min(FB, n - k0);
    for (int i = 0; i < FB; ++i) sD[i][lane] = (i < kb && lane < kb) ? A[(size_t)(k0 + i) * ld + k0 + lane] : (i == lane ? 1.0 : 0.0);
    __syncwarp();
    bool fail = false;
    for (int j = 0; j < kb; ++j) {                              // left-looking, lane = row (as in chol_kernel)
        double v = sD[lane][j];
        for (int k = 0; k < j; ++k) v = fma(-sD[lane][k], sD[j][k], v);
        double piv = __shfl_sync(0xffffffffu, v, j);
        if (!(piv > 0.0)) { fail = true; piv = 1.0; }
        const double rp = 1.0 / sqrt(piv);
        __syncwarp();
        if (lane >= j) sD[lane][j] = (lane == j) ? sqrt(piv) : v * rp;
        __syncwarp();
    }
    for (int i = 0; i < kb; ++i) if (lane < kb) A[(size_t)(k0 + i) * ld + k0 + lane] = (lane <= i) ? sD[i][lane] : 0.0;
    if (lane == 0 && fail && info) atomicOr(&info[blockIdx.x / mats_per_b], 2);
}
__global__ void __launch_bounds__(256) chol_panel_kernel(int n, int k0, double* Aall, int ld, long long ms) {
    PDL_ENTRY();
    __shared__ double sD[FB][FB + 1];
    double* A = Aall + (size_t)blockIdx.y * ms;
    const int tid = threadIdx.x, kb = min(FB, n - k0);
    for (int e = tid; e < FB * FB; e += 256) {
        const int i = e / FB, j = e % FB;
        sD[i][j] = (i < kb && j < kb) ? A[(size_t)(k0 + i) * ld + k0 + j] : (i == j ? 1.0 : 0.0);
    }
    __syncthreads();
    const int i = k0 + kb + blockIdx.x * 256 + tid;
    if (i >= n) return;
    double x[FB];
    double* arow = A + (size_t)i * ld + k0;
#pragma unroll
    for (int j = 0; j < FB; ++j) x[j] = j < kb ? arow[j] : 0.0;
#pragma unroll
    for (int j = 0; j < FB; ++j) {
        if (j < kb) {
            double v = x[j];
#pragma unroll
            for (int k = 0; k < j; ++k) v = fma(-x[k], sD[j][k], v);
            x[j] = v / sD[j][j];
        }
    }
#pragma unroll
    for (int j = 0; j < FB; ++j) if (j < kb) arow[j] = x[j];
}
__global__ void __launch_bounds__(256) chol_kernel(int n, double* Aall, int ld, long long ms, int mats_per_b, int* info);
// in-place lower Cholesky of `batch` matrices (info index = matrix / mats_per_b): one CTA per matrix when small
static int chol_launch(cudaStream_t st, int batch, int n, double* A, int ld, long long ms, int mats_per_b, int* info) {
    static int single = -1;                                     // PILCO_CHOL_SINGLE=1: always the one-CTA kernel (A/B switch)
    if (single < 0) { const char* e = getenv("PILCO_CHOL_SINGLE"); single = (e && e[0] == '1') ? 1 : 0; }
    if (n < CHOL_MULTI_N || single) {
        launch_hi(chol_kernel, dim3(batch), dim3(256), 0, st, n, A, ld, ms, mats_per_b, info);
        CUDA_LAUNCH_CHECK();
        return PILCO_OK;
    }
    for (int k0 = 0; k0 < n; k0 += FB) {
        const int kb = min(FB, n - k0), t0 = k0 + kb;
        launch_hi(chol_diag_kernel, dim3(batch), dim3(32), 0, st, n, k0, A, ld, ms, mats_per_b, info);
        if (t0 >= n) break;
        launch_hi(chol_panel_kernel, dim3((n - t0 + 255) / 256, batch), dim3(256), 0, st, n, k0, A, ld, ms);
        CUDA_LAUNCH_CHECK();
        const double* P = A + (size_t)t0 * ld + k0;              // L21 [n - t0, kb]
        int rc = gemm(st, batch, n - t0, n - t0, kb, 0, 1, -1.0, P, ld, ms, P, ld, ms, 1.0, A + (size_t)t0 * ld + t0, ld, ms);
        if (rc) return rc;
    }
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

// X = L^-1 (lower triangular), X zero-initialised by the caller outside the diagonal blocks.
// T: scratch [batch, FB, ld]
static int tri_inverse(cudaStream_t st, int batch, int n, const double* L, int ld, long long ms,
                       double* X, int ldx, long long xs, double* T, long long ts) {
    const int nb = (n + FB - 1) / FB;
    tri_diag_inv_kernel<<<dim3(nb, batch), 32, 0, st>>>(n, L, ld, ms, X, ldx, xs);
    CUDA_LAUNCH_CHECK();
    for (int I = 1; I < nb; ++I) {
        const int r0 = I * FB, rb = min(FB, n - r0);
        // T = L[I, 0:r0] X[0:r0, 0:r0]
        int rc = gemm(st, batch, rb, r0, r0, 0, 0, 1.0, L + (size_t)r0 * ld, ld, ms, X, ldx, xs, 0.0, T, ld, ts);
        if (rc) return rc;
        // X[I, 0:r0] = -X_II T
        rc = gemm(st, batch, rb, r0, rb, 0, 0, -1.0, X + (size_t)r0 * ldx + r0, ldx, xs, T, ld, ts, 0.0,
                  X + (size_t)r0 * ldx, ldx, xs);
        if (rc) return rc;
    }
    return PILCO_OK;
}

// -------------------------------------------------------------------------------------------------
// small helpers
// -------------------------------------------------------------------------------------------------
// y[z][i] = sum_j op(A[z])[i][j] x[z][j]   (one warp per row; grid (m, batch))
__global__ void __launch_bounds__(32) matvec_kernel(int m, int k, int ta, const double* A, int lda, long long sa,
                                                    const double* x, long long xs, int xinc,
                                                    double* y, long long ys) {
    const int i = blockIdx.x, z = blockIdx.y, lane = threadIdx.x;
    const double* Az = A + (size_t)z * sa;
    const double* xz = x + (size_t)z * xs;
    double v = 0.0;
    for (int j = lane; j < k; j += 32) v = fma(ta ? Az[(size_t)j * lda + i] : Az[(size_t)i * lda + j], xz[(size_t)j * xinc], v);
    v = warp_sum(v);
    if (lane == 0) y[(size_t)z * ys + i] = v;
}

// Solve L L^T x = y for one right-hand side per matrix by blocked substitution (one CTA per matrix).
// L lower triangular [n,n] (ld), y stride yinc, x contiguous [n].
// Matrix z = b*E + e takes its right-hand side at Y + b*Y_bs + e*y_es with element increment yinc
// (column e of an [n,E] array: y_es=1, yinc=E; row e of an [E,n] array: y_es=n, yinc=1).
__global__ void __launch_bounds__(256) chol_solve_vec_kernel(int n, const double* Lall, int ld, long long ms,
                                                             int E, const double* Y, long long Y_bs,
                                                             long long y_es, int yinc,
                                                             double* xall, long long xs) {
    PDL_ENTRY();
    extern __shared__ double sx[];            // n doubles
    __shared__ double sD[FB][FB + 1];
    const double* L = Lall + (size_t)blockIdx.x * ms;
    const double* y = Y + (size_t)(blockIdx.x / E) * Y_bs + (size_t)(blockIdx.x % E) * y_es;
    double* x = xall + (size_t)blockIdx.x * xs;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < n; i += 256) sx[i] = y[(size_t)i * yinc];
    __syncthreads();
    const int nb = (n + FB - 1) / FB;
    for (int I = 0; I < nb; ++I) {                                   // forward  L z = y
        const int r0 = I * FB, rb = min(FB, n - r0);
        for (int rr = warp; rr < rb; rr += 8) {                      // sx[r0+rr] -= L[r0+rr, 0:r0] . sx[0:r0]
            double v = 0.0;
            for (int k = lane; k < r0; k += 32) v = fma(L[(size_t)(r0 + rr) * ld + k], sx[k], v);
            v = warp_sum(v);
            if (lane == 0) sx[r0 + rr] -= v;
        }
        for (int e = tid; e < FB * FB; e += 256) {
            const int i = e / FB, j = e % FB;
            sD[i][j] = (i < rb && j < rb) ? L[(size_t)(r0 + i) * ld + r0 + j] : (i == j ? 1.0 : 0.0);
        }
        __syncthreads();
        if (tid == 0) {
            for (int i = 0; i < rb; ++i) {
                double v = sx[r0 + i];
                for (int k = 0; k < i; ++k) v = fma(-sD[i][k], sx[r0 + k], v);
                sx[r0 + i] = v / sD[i][i];
            }
        }
        __syncthreads();
    }
    for (int I = nb - 1; I >= 0; --I) {                              // backward  L^T x = z
        const int r0 = I * FB, rb = min(FB, n - r0);
        for (int rr = warp; rr < rb; rr += 8) {                      // sx[r0+rr] -= L[r1:, r0+rr] . sx[r1:]
            double v = 0.0;
            for (int k = r0 + rb + lane; k < n; k += 32) v = fma(L[(size_t)k * ld + r0 + rr], sx[k], v);
            v = warp_sum(v);
            if (lane == 0) sx[r0 + rr] -= v;
        }
        for (int e = tid; e < FB * FB; e += 256) {
            const int i = e / FB, j = e % FB;
            sD[i][j] = (i < rb && j < rb) ? L[(size_t)(r0 + i) * ld + r0 + j] : (i == j ? 1.0 : 0.0);
        }
        __syncthreads();
        if (tid == 0) {
            for (int i = rb - 1; i >= 0; --i) {
                double v = sx[r0 + i];
                for (int k = i + 1; k < rb; ++k) v = fma(-sD[k][i], sx[r0 + k], v);
                sx[r0 + i] = v / sD[i][i];
            }
        }
        __syncthreads();
    }
    for (int i = tid; i < n; i += 256) x[i] = sx[i];
}

__global__ void fill_kernel(double* p, size_t count, double v) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}
static void fill(cudaStream_t st, double* p, size_t count, double v) {
    if (count == 0) return;
    if (v == 0.0) { cudaMemsetAsync(p, 0, count * sizeof(double), st); return; }
    fill_kernel<<<(unsigned)min((size_t)1024, (count + 255) / 256), 256, 0, st>>>(p, count, v);
}

// FITC: G[j] = sqrt(1 + (sf2 - sum_i V[i][j]^2)/sn2);  V[:,j] /= G[j];  Vg = V/G (second division)
__global__ void fitc_scale_kernel(int Mi, int N, double* V, int ldv, long long vs, double* Vg, const double* sf2,
                                  const double* sn2) {
    const int e = blockIdx.y;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    double* Ve = V + (size_t)e * vs;
    double* Vge = Vg + (size_t)e * vs;
    double ss = 0.0;
    for (int i = 0; i < Mi; ++i) { const double v = Ve[(size_t)i * ldv + j]; ss = fma(v, v, ss); }
    const double G = sqrt(1.0 + (sf2[e] - ss) / sn2[e]);
    for (int i = 0; i < Mi; ++i) {
        const double v = Ve[(size_t)i * ldv + j] / G;
        Ve[(size_t)i * ldv + j] = v;
        Vge[(size_t)i * ldv + j] = v / G;
    }
}

__global__ void add_diag_kernel(int n, double* A, int ld, long long ms, const double* d) {
    const int e = blockIdx.y;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(size_t)e * ms + (size_t)i * ld + i] += d[e];
}

__global__ void fitc_axpy_kernel(int n, double* C, int ldc, long long cs, const double* Tm, int ldt, long long ts, const double* a) {
    const int e = blockIdx.z, j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i < n && j < n) C[(size_t)e * cs + (size_t)i * ldc + j] -= a[e] * Tm[(size_t)e * ts + (size_t)i * ldt + j];
}

void chol_solve_vec_launch(cudaStream_t st, int batch, int n, const double* L, int ld, long long ms, int E,
                           const double* Y, long long Y_bs, long long y_es, int yinc, double* x, long long xs) {
    launch_hi(chol_solve_vec_kernel, dim3(batch), dim3(256), n * sizeof(double), st, n, L, ld, ms, E, Y, Y_bs, y_es, yinc, x, xs);
}

extern "C" {

size_t pilco_gp_factorize_workspace_bytes(int n, int E, int B) {
    if (n < 1 || E < 1 || B < 1) return 0;
    const size_t ldk = pad64(n);
    return ((size_t)B * E * (2 * ldk * ldk + FB * ldk)) * sizeof(double);
}

int pilco_gp_factorize(int n, int D, int E, int B,
                       const double* X, long long X_bs, const double* Y, long long Y_bs,
                       const double* ell, long long ell_bs, const double* sf2, long long sf2_bs,
                       const double* sn2, long long sn2_bs,
                       double* iK, int ldk, double* beta, int* info,
                       void* ws, size_t ws_bytes, pilco_stream_t stream) {
    if (!X || !Y || !ell || !sf2 || !sn2 || !beta || !ws) return PILCO_ERR_NULL;
    if (n < 1 || D < 1 || D > MAXD || E < 1 || E > MAXE || B < 1) return PILCO_ERR_DIM;
    if (iK && ldk < pad64(n)) return PILCO_ERR_DIM;
    if (ws_bytes < pilco_gp_factorize_workspace_bytes(n, E, B)) return PILCO_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int ldw = pad64(n);
    const long long ms = (long long)ldw * ldw;
    const int batch = B * E;
    double* L = (double*)ws;
    double* Xi = L + (size_t)batch * ms;
    double* T = Xi + (size_t)batch * ms;
    if (info) cudaMemsetAsync(info, 0, sizeof(int) * B, st);
    // K + sn2 I  (mgpr.py:82-84), zero outside n x n
    GramArgs g{n, n, D, E, X, X_bs, X, X_bs, ell, ell_bs, sf2, sf2_bs, sn2, sn2_bs, 0.0, L, ldw, ms, ldw, ldw, 0};
    launch_hi(gram_kernel, dim3((ldw + 31) / 32, (ldw + 7) / 8, batch), dim3(32, 8), 0, st, g);
    CUDA_LAUNCH_CHECK();
    { int rcc = chol_launch(st, batch, n, L, ldw, ms, E, info); if (rcc) return rcc; }
    CUDA_LAUNCH_CHECK();
    // beta = (L L^T)^-1 y_e   (mgpr.py:86-88)
    launch_hi(chol_solve_vec_kernel, dim3(batch), dim3(256), n * sizeof(double), st, n, L, ldw, ms, E, Y, Y_bs, 1, E, beta, n);
    CUDA_LAUNCH_CHECK();
    if (iK) {
        // iK = L^-T L^-1 through the explicit triangular inverse (mgpr.py:85)
        cudaMemsetAsync(Xi, 0, (size_t)batch * ms * sizeof(double), st);
        int rc = tri_inverse(st, batch, n, L, ldw, ms, Xi, ldw, ms, T, (long long)FB * ldw);
        if (rc) return rc;
        cudaMemsetAsync(iK, 0, (size_t)batch * ldk * ldk * sizeof(double), st);
        rc = gemm(st, batch, n, n, n, 1, 0, 1.0, Xi, ldw, ms, Xi, ldw, ms, 0.0, iK, ldk, (long long)ldk * ldk);
        if (rc) return rc;
    }
    return PILCO_OK;
}

// ---- incremental set_data: k rows appended to a factorised model, hyper-parameters unchanged -------------------
// (SURVEY section 8f-2; pilco/models/mgpr.py:38-45 swaps the data, examples/inv_double_pendulum.py:102-103 and
// swimmer.py:87-88 append the T rows of every new episode).  Block inverse of A1 = [[A0, K12], [K21, K22 + sn2 I]]:
//   F = K21 A0^-1,  S = K22 + sn2 I - F K12 (Schur complement, k x k, SPD),  G = S^-1 F,
//   A1^-1 = [[A0^-1 + F' G, -G'], [-G, S^-1]],   beta = A1^-1 y.
// O(n^2 k) instead of O(n^3); only the old inverse is needed (no Cholesky factor of the old matrix).
__global__ void __launch_bounds__(256) append_assemble_kernel(int n0, int k, const double* G, int ldg, long long gs,
                                                              const double* Sinv, int lds, long long ss,
                                                              double* iK, int ldk, long long ks) {
    PDL_ENTRY();
    const int e = blockIdx.y;
    const int n1 = n0 + k;
    const double* Ge = G + (size_t)e * gs;
    const double* Se = Sinv + (size_t)e * ss;
    double* O = iK + (size_t)e * ks;
    for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < (size_t)k * n1; idx += (size_t)gridDim.x * blockDim.x) {
        const int i = (int)(idx / n1), j = (int)(idx % n1);          // row n0 + i of the new inverse
        if (j < n0) {
            const double v = -Ge[(size_t)i * ldg + j];
            O[(size_t)(n0 + i) * ldk + j] = v;
            O[(size_t)j * ldk + n0 + i] = v;
        } else {
            O[(size_t)(n0 + i) * ldk + j] = Se[(size_t)i * lds + (j - n0)];
        }
    }
}

extern "C" size_t pilco_gp_append_workspace_bytes(int n0, int k, int E) {
    if (n0 < 1 || k < 1 || E < 1) return 0;
    const size_t ld0 = pad64(n0), kp = pad64(k);
    // K21, F, G: [kp x ld0] each; S, L^-1, S^-1: [kp x kp]; T: [FB x kp]
    return (size_t)E * (3 * kp * ld0 + 3 * kp * kp + FB * kp) * sizeof(double);
}

extern "C" int pilco_gp_append(int n0, int k, int D, int E,
                               const double* X, const double* Y,            /* [n0+k, D], [n0+k, E]: old rows first */
                               const double* ell, const double* sf2, const double* sn2,
                               const double* iK_old, int ldk_old,
                               double* iK_new, int ldk_new, double* beta_new, int* info,
                               void* ws, size_t ws_bytes, pilco_stream_t stream) {
    if (!X || !Y || !ell || !sf2 || !sn2 || !iK_old || !iK_new || !beta_new || !ws) return PILCO_ERR_NULL;
    if (n0 < 1 || k < 1 || D < 1 || D > MAXD || E < 1 || E > MAXE) return PILCO_ERR_DIM;
    const int n1 = n0 + k;
    if (ldk_old < pad64(n0) || ldk_new < pad64(n1)) return PILCO_ERR_DIM;
    if (iK_old == iK_new) return PILCO_ERR_DIM;                             // out of place (leading dimensions may differ)
    if (ws_bytes < pilco_gp_append_workspace_bytes(n0, k, E)) return PILCO_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int ld0 = pad64(n0), kp = pad64(k);
    const long long rs = (long long)kp * ld0, qs = (long long)kp * kp;
    double* K21 = (double*)ws;
    double* F = K21 + (size_t)E * rs;
    double* G = F + (size_t)E * rs;
    double* S = G + (size_t)E * rs;
    double* Li = S + (size_t)E * qs;
    double* Si = Li + (size_t)E * qs;
    double* T = Si + (size_t)E * qs;
    const double* Xn = X + (size_t)n0 * D;
    if (info) cudaMemsetAsync(info, 0, sizeof(int), st);
    // K21 = k(Xnew, Xold) [k x n0];  S = k(Xnew, Xnew) + sn2 I
    GramArgs g1{k, n0, D, E, Xn, 0, X, 0, ell, 0, sf2, 0, nullptr, 0, 0.0, K21, ld0, rs, k, n0, 0};
    launch_hi(gram_kernel, dim3((n0 + 31) / 32, (k + 7) / 8, E), dim3(32, 8), 0, st, g1);
    GramArgs g2{k, k, D, E, Xn, 0, Xn, 0, ell, 0, sf2, 0, sn2, 0, 0.0, S, kp, qs, kp, kp, 0};
    launch_hi(gram_kernel, dim3((kp + 31) / 32, (kp + 7) / 8, E), dim3(32, 8), 0, st, g2);
    CUDA_LAUNCH_CHECK();
    const long long ko = (long long)ldk_old * ldk_old, kn = (long long)ldk_new * ldk_new;
    int rc = gemm(st, E, k, n0, n0, 0, 0, 1.0, K21, ld0, rs, iK_old, ldk_old, ko, 0.0, F, ld0, rs);          // F = K21 A0^-1
    if (rc) return rc;
    rc = gemm(st, E, k, k, n0, 0, 1, -1.0, F, ld0, rs, K21, ld0, rs, 1.0, S, kp, qs);                        // S -= F K12
    if (rc) return rc;
    { int rcc = chol_launch(st, E, k, S, kp, qs, E, info); if (rcc) return rcc; }
    CUDA_LAUNCH_CHECK();
    cudaMemsetAsync(Li, 0, (size_t)E * qs * sizeof(double), st);
    rc = tri_inverse(st, E, k, S, kp, qs, Li, kp, qs, T, (long long)FB * kp);
    if (rc) return rc;
    rc = gemm(st, E, k, k, k, 1, 0, 1.0, Li, kp, qs, Li, kp, qs, 0.0, Si, kp, qs);                           // S^-1 = L^-T L^-1
    if (rc) return rc;
    rc = gemm(st, E, k, n0, k, 0, 0, 1.0, Si, kp, qs, F, ld0, rs, 0.0, G, ld0, rs);                          // G = S^-1 F
    if (rc) return rc;
    // new inverse: zero padded [ldk_new x ldk_new]; old block copied, then + F' G; then the border blocks
    cudaMemsetAsync(iK_new, 0, (size_t)E * kn * sizeof(double), st);
    for (int e = 0; e < E; ++e)
        cudaMemcpy2DAsync(iK_new + (size_t)e * kn, (size_t)ldk_new * sizeof(double), iK_old + (size_t)e * ko,
                          (size_t)ldk_old * sizeof(double), (size_t)n0 * sizeof(double), n0, cudaMemcpyDeviceToDevice, st);
    rc = gemm(st, E, n0, n0, k, 1, 0, 1.0, F, ld0, rs, G, ld0, rs, 1.0, iK_new, ldk_new, kn);
    if (rc) return rc;
    launch_hi(append_assemble_kernel, dim3((unsigned)min((size_t)256, ((size_t)k * n1 + 255) / 256), E), dim3(256), 0, st,
              n0, k, (const double*)G, ld0, rs, (const double*)Si, kp, qs, iK_new, ldk_new, kn);
    CUDA_LAUNCH_CHECK();
    // beta = A1^-1 y_e  (row e of beta [E, n1]; y_e = column e of Y)
    matvec_kernel<<<dim3(n1, E), 32, 0, st>>>(n1, n1, 0, iK_new, ldk_new, kn, Y, 1, E, beta_new, n1);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

// ---- GP training objective: -log p(y | X, theta) and its gradient w.r.t. (ell, sf2, sn2) ------------------------
// Replaces gpflow.models.GPR.training_loss + TF autodiff as used by MGPR.optimize (pilco/models/mgpr.py:47-75;
// priors are added on the host).  d/dtheta = -0.5 tr((alpha alpha^T - K^-1) dK/dtheta).
__global__ void __launch_bounds__(256) gp_nlml_grad_kernel(int n, int D, int E, const double* X, long long X_bs,
                                                           const double* Y, long long Y_bs,
                                                           const double* ell, long long ell_bs,
                                                           const double* sf2, long long sf2_bs,
                                                           const double* Lall, const double* iKall, int ldw,
                                                           const double* alpha,
                                                           double* nlml, double* g_ell, double* g_sf2, double* g_sn2) {
    const int z = blockIdx.x, bidx = z / E, e = z % E;
    const int tid = threadIdx.x;
    const double* Xb = X + (size_t)bidx * X_bs;
    const double* Yb = Y + (size_t)bidx * Y_bs;
    const double* le = ell + (size_t)bidx * ell_bs + (size_t)e * D;
    const double sf = sf2[(size_t)bidx * sf2_bs + e];
    const double* L = Lall + (size_t)z * ldw * ldw;
    const double* iK = iKall + (size_t)z * ldw * ldw;
    const double* al = alpha + (size_t)z * n;
    __shared__ double sred[(MAXD + 4) * 8], sout[MAXD + 4];
    double il[MAXD];
#pragma unroll
    for (int d = 0; d < MAXD; ++d) il[d] = d < D ? 1.0 / le[d] : 0.0;
    double acc[MAXD + 3];                    // [0..D): ell, [MAXD]: sf2, [MAXD+1]: sn2, [MAXD+2]: nlml pieces
#pragma unroll
    for (int i = 0; i < MAXD + 3; ++i) acc[i] = 0.0;
    for (int idx = tid; idx < n * n; idx += blockDim.x) {
        const int i = idx / n, j = idx % n;
        double d2 = 0.0, df[MAXD];
#pragma unroll
        for (int d = 0; d < MAXD; ++d) {
            df[d] = d < D ? (Xb[(size_t)i * D + d] - Xb[(size_t)j * D + d]) * il[d] : 0.0;
            d2 = fma(df[d], df[d], d2);
        }
        const double Kf = sf * exp(-0.5 * d2);
        const double W = al[i] * al[j] - iK[(size_t)i * ldw + j];
        const double t = W * Kf;
        acc[MAXD] += t;
#pragma unroll
        for (int d = 0; d < MAXD; ++d) acc[d] = fma(t, df[d] * df[d], acc[d]);    // (x_i-x_j)^2/ell^2 ; /ell below
        if (i == j) acc[MAXD + 1] += W;
    }
    for (int i = tid; i < n; i += blockDim.x)
        acc[MAXD + 2] += 0.5 * Yb[(size_t)i * E + e] * al[i] + log(L[(size_t)i * ldw + i]);
    block_sum<MAXD + 3>(acc, MAXD + 3, sred, sout);
    if (tid < D) g_ell[(size_t)z * D + tid] = -0.5 * sout[tid] * il[tid];       // dK/dell_d = K (x-x')^2 / ell^3
    if (tid == 0) {
        g_sf2[z] = -0.5 * sout[MAXD] / sf;
        g_sn2[z] = -0.5 * sout[MAXD + 1];
        nlml[z] = sout[MAXD + 2] + 0.5 * n * 1.8378770664093453;               // log(2 pi)
    }
}

size_t pilco_gp_nlml_workspace_bytes(int n, int E, int B) {
    if (n < 1 || E < 1 || B < 1) return 0;
    const size_t ldw = pad64(n);
    return pilco_gp_factorize_workspace_bytes(n, E, B) + ((size_t)B * E * (ldw * ldw + ldw)) * sizeof(double);
}

int pilco_gp_nlml(int n, int D, int E, int B,
                  const double* X, long long X_bs, const double* Y, long long Y_bs,
                  const double* ell, long long ell_bs, const double* sf2, long long sf2_bs,
                  const double* sn2, long long sn2_bs,
                  double* nlml, double* g_ell, double* g_sf2, double* g_sn2, int* info,
                  void* ws, size_t ws_bytes, pilco_stream_t stream) {
    if (!nlml || !g_ell || !g_sf2 || !g_sn2 || !ws) return PILCO_ERR_NULL;
    if (ws_bytes < pilco_gp_nlml_workspace_bytes(n, E, B)) return PILCO_ERR_WORKSPACE;
    const size_t fbytes = pilco_gp_factorize_workspace_bytes(n, E, B);
    const int ldw = pad64(n);
    double* fws = (double*)ws;
    double* iK = (double*)((char*)ws + fbytes);
    double* alpha = iK + (size_t)B * E * ldw * ldw;
    int rc = pilco_gp_factorize(n, D, E, B, X, X_bs, Y, Y_bs, ell, ell_bs, sf2, sf2_bs, sn2, sn2_bs,
                                iK, ldw, alpha, info, fws, fbytes, stream);
    if (rc) return rc;
    gp_nlml_grad_kernel<<<B * E, 256, 0, (cudaStream_t)stream>>>(n, D, E, X, X_bs, Y, Y_bs, ell, ell_bs, sf2, sf2_bs,
                                                                 fws, iK, ldw, alpha, nlml, g_ell, g_sf2, g_sn2);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

// ---- FITC training objective on the device (SURVEY section 8f-1, second half) -----------------------------------
// Replaces gpflow.models.GPRFITC.training_loss + TF autodiff as used by SMGPR.optimize (pilco/models/smgpr.py:16-22 via
// mgpr.py:47-75): value and gradient w.r.t. (ell, sf2, sn2, Z) of the collapsed FITC bound, batched over
// B hyper-parameter sets x E outputs (every output trains its own inducing inputs Z).  Stage by stage the algorithm of
// oracle/fitc_staged.py (checked against torch autograd there):
//   Kuf, Kuu -> Luu = chol(Kuu + 1e-6 I) -> V = Luu^-1 Kuf -> nu = sf2 + sn2 - colsum(V o V) -> B = I + V diag(1/nu) V'
//   -> L = chol(B) -> alpha = V (y/nu), gamma = L^-1 alpha -> value;   reverse sweep with two Cholesky adjoints
//   (Kbar = sym(L^-T Phi(L' Lbar) L^-1)) and the SE-ARD kernel adjoints.  All N-sized products are GEMMs (gemm_kernel).
struct FitcWs { size_t Kuf, V, T1, T2, Kuu0, Luu, LinvU, Bm, LinvB, Pm, Qm, Ts, nu, ynu, nub, al, ga, ab, part, per_z; };
static FitcWs fitc_ws_layout(int N, int Mi, int D) {
    FitcWs W; size_t o = 0;
    const size_t ldm = pad64(Mi), ldn = pad64(N);
    auto take = [&](size_t len) { size_t at = o; o += (len + 1) & ~(size_t)1; return at; };
    W.Kuf = take(ldm * ldn); W.V = take(ldm * ldn); W.T1 = take(ldm * ldn); W.T2 = take(ldm * ldn);
    W.Kuu0 = take(ldm * ldm); W.Luu = take(ldm * ldm); W.LinvU = take(ldm * ldm); W.Bm = take(ldm * ldm);
    W.LinvB = take(ldm * ldm); W.Pm = take(ldm * ldm); W.Qm = take(ldm * ldm); W.Ts = take(ldm * ldm);
    W.nu = take(ldn); W.ynu = take(ldn); W.nub = take(ldn);
    W.al = take(ldm); W.ga = take(ldm); W.ab = take(ldm);
    W.part = take((size_t)Mi * (MAXD + 2));
    W.per_z = o;
    return W;
}

// per column n: nu, y/nu and Vs = V / nu
__global__ void fitc_nu_kernel(int Mi, int N, int E, const double* V, int ldn, long long zs, const double* Y,
                               const double* sf2, const double* sn2, double* Vs, double* nu, double* ynu) {
    const int z = blockIdx.y, e = z % E;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const double* Vz = V + (size_t)z * zs + n;
    double ss = 0.0;
    for (int i = 0; i < Mi; ++i) { const double v = Vz[(size_t)i * ldn]; ss = fma(v, v, ss); }
    const double nv = sf2[z] + sn2[z] - ss;
    nu[(size_t)z * zs + n] = nv;
    ynu[(size_t)z * zs + n] = Y[(size_t)n * E + e] / nv;
    double* Vsz = Vs + (size_t)z * zs + n;
    for (int i = 0; i < Mi; ++i) Vsz[(size_t)i * ldn] = Vz[(size_t)i * ldn] / nv;
}
// (the three vectors above live in the per-z workspace: same stride zs as the matrices)

__global__ void add_diag_const_kernel(int n, double* A, int ld, long long ms, double c) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) A[(size_t)blockIdx.y * ms + (size_t)i * ld + i] += c;
}

// Pm = tril(Lbar), Lbar = ab gamma' + diag(1 / L_ii)      (Lbar of the value w.r.t. L = chol(B))
__global__ void fitc_lbar_kernel(int Mi, const double* L, int ld, long long zs, const double* ab, const double* ga, double* Pm) {
    const int z = blockIdx.z, j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= Mi || j >= Mi) return;
    double v = 0.0;
    if (j <= i) {
        v = ab[(size_t)z * zs + i] * ga[(size_t)z * zs + j];
        if (i == j) v += 1.0 / L[(size_t)z * zs + (size_t)i * ld + i];
    }
    Pm[(size_t)z * zs + (size_t)i * ld + j] = v;
}
// mode 0: zero the strict upper triangle;  1: Phi (lower triangle, diagonal halved);  2: symmetrise
__global__ void tri_op_kernel(int n, double* A, int ld, long long zs, int mode) {
    const int z = blockIdx.z, j = blockIdx.x * 32 + threadIdx.x, i = blockIdx.y * 8 + threadIdx.y;
    if (i >= n || j >= n) return;
    double* Az = A + (size_t)z * zs;
    if (mode == 2) { if (j < i) { const double v = 0.5 * (Az[(size_t)i * ld + j] + Az[(size_t)j * ld + i]); Az[(size_t)i * ld + j] = v; Az[(size_t)j * ld + i] = v; } return; }
    if (j > i) Az[(size_t)i * ld + j] = 0.0;
    else if (mode == 1 && i == j) Az[(size_t)i * ld + j] *= 0.5;
}
// per column n:  nu_bar and V_bar (in place over BV)
__global__ void fitc_cols_bwd_kernel(int Mi, int N, int E, const double* V, double* BV, int ldn, long long zs, const double* Y,
                                     const double* nu, const double* ynu, const double* ab, double* nub) {
    const int z = blockIdx.y, e = z % E;
    const int n = blockIdx.x * blockDim.x + threadIdx.x;
    if (n >= N) return;
    const double* Vz = V + (size_t)z * zs + n;
    double* Bz = BV + (size_t)z * zs + n;
    const double* abz = ab + (size_t)z * zs;
    double s1 = 0.0, a = 0.0;
    for (int i = 0; i < Mi; ++i) { const double v = Vz[(size_t)i * ldn]; s1 = fma(v, Bz[(size_t)i * ldn], s1); a = fma(abz[i], v, a); }
    const double nv = nu[(size_t)z * zs + n], y = Y[(size_t)n * E + e], in2 = 1.0 / (nv * nv);
    const double nb = -s1 * in2 + a * y * in2 - 0.5 * y * y * in2 + 0.5 / nv;     // (alpha_bar = -ab)
    nub[(size_t)z * zs + n] = nb;
    const double yn = ynu[(size_t)z * zs + n];
    for (int i = 0; i < Mi; ++i)
        Bz[(size_t)i * ldn] = 2.0 * Bz[(size_t)i * ldn] / nv - abz[i] * yn - 2.0 * Vz[(size_t)i * ldn] * nb;
}
// kernel adjoints, one CTA per (z, inducing point i):  Guf = Kuf_bar o Kuf (row i), Guu = Kuu_bar o Kuu (row i, symmetric)
//   gZ[i,d] = -( sum_n Guf (z_id - x_nd) + 2 sum_j Guu (z_id - z_jd) ) / ell_d^2
//   part[i] = [ sum_n Guf dzx_d^2 + sum_j Guu dzz_d^2  (d < D) | sum Guf + sum Guu ]
__global__ void __launch_bounds__(128) fitc_adjoint_kernel(int Mi, int N, int D, const double* X, const double* Z, const double* ell,
                                                           const double* Kuf, const double* Kufb, int ldn,
                                                           const double* Kuu0, const double* Kuub, int ldm, long long zs,
                                                           double* part, double* gZ) {
    const int z = blockIdx.y, i = blockIdx.x, tid = threadIdx.x;
    const double* Zz = Z + (size_t)z * Mi * D;
    __shared__ double sred[(2 * MAXD + 1) * 4], sout[2 * MAXD + 1];
    double zi[MAXD], acc[2 * MAXD + 1];
#pragma unroll
    for (int d = 0; d < MAXD; ++d) zi[d] = d < D ? Zz[(size_t)i * D + d] : 0.0;
#pragma unroll
    for (int k = 0; k < 2 * MAXD + 1; ++k) acc[k] = 0.0;
    const double* kf = Kuf + (size_t)z * zs + (size_t)i * ldn;
    const double* kb = Kufb + (size_t)z * zs + (size_t)i * ldn;
    for (int n = tid; n < N; n += blockDim.x) {
        const double gq = kf[n] * kb[n];
        acc[2 * MAXD] += gq;
#pragma unroll
        for (int d = 0; d < MAXD; ++d) if (d < D) { const double df = zi[d] - X[(size_t)n * D + d]; acc[d] = fma(gq, df, acc[d]); acc[MAXD + d] = fma(gq * df, df, acc[MAXD + d]); }
    }
    const double* ku = Kuu0 + (size_t)z * zs + (size_t)i * ldm;
    const double* kub = Kuub + (size_t)z * zs + (size_t)i * ldm;
    for (int j = tid; j < Mi; j += blockDim.x) {
        const double gq = ku[j] * kub[j];
        acc[2 * MAXD] += gq;
#pragma unroll
        for (int d = 0; d < MAXD; ++d) if (d < D) { const double df = zi[d] - Zz[(size_t)j * D + d]; acc[d] = fma(2.0 * gq, df, acc[d]); acc[MAXD + d] = fma(gq * df, df, acc[MAXD + d]); }
    }
    block_sum<2 * MAXD + 1>(acc, 2 * MAXD + 1, sred, sout);
    if (tid < D) {
        const double l = ell[(size_t)z * D + tid];
        gZ[((size_t)z * Mi + i) * D + tid] = -sout[tid] / (l * l);
        part[(size_t)z * zs + (size_t)i * (MAXD + 2) + tid] = sout[MAXD + tid];
    }
    if (tid == 0) part[(size_t)z * zs + (size_t)i * (MAXD + 2) + MAXD] = sout[2 * MAXD];
}
// value and the remaining gradients of one (b, e)
__global__ void __launch_bounds__(256) fitc_final_kernel(int Mi, int N, int D, int E, const double* Y, const double* ell, const double* sf2,
                                                         const double* L, int ldm, const double* nu, const double* nub, const double* ga,
                                                         const double* part, long long zs,
                                                         double* nlml, double* g_ell, double* g_sf2, double* g_sn2) {
    const int z = blockIdx.x, e = z % E, tid = threadIdx.x;
    __shared__ double sred[(MAXD + 4) * 8], sout[MAXD + 4];
    double acc[MAXD + 4];                     // [0..D): ell pieces, [MAXD]: sum G, [MAXD+1]: sum nu_bar, [MAXD+2]: value pieces
#pragma unroll
    for (int k = 0; k < MAXD + 4; ++k) acc[k] = 0.0;
    for (int n = tid; n < N; n += blockDim.x) {
        const double nv = nu[(size_t)z * zs + n], y = Y[(size_t)n * E + e];
        acc[MAXD + 1] += nub[(size_t)z * zs + n];
        acc[MAXD + 2] += 0.5 * y * y / nv + 0.5 * log(nv);
    }
    for (int i = tid; i < Mi; i += blockDim.x) {
        const double g = ga[(size_t)z * zs + i];
        acc[MAXD + 2] += -0.5 * g * g + log(L[(size_t)z * zs + (size_t)i * ldm + i]);
        const double* pr = part + (size_t)z * zs + (size_t)i * (MAXD + 2);
#pragma unroll
        for (int d = 0; d < MAXD; ++d) if (d < D) acc[d] += pr[d];
        acc[MAXD] += pr[MAXD];
    }
    block_sum<MAXD + 4>(acc, MAXD + 4, sred, sout);
    if (tid < D) { const double l = ell[(size_t)z * D + tid]; g_ell[(size_t)z * D + tid] = sout[tid] / (l * l * l); }
    if (tid == 0) {
        nlml[z] = sout[MAXD + 2] + 0.5 * N * 1.8378770664093453;            // log(2 pi)
        g_sf2[z] = sout[MAXD + 1] + sout[MAXD] / sf2[z];
        g_sn2[z] = sout[MAXD + 1];
    }
}

size_t pilco_fitc_nlml_workspace_bytes(int N, int Mi, int D, int E, int B) {
    if (N < 1 || Mi < 1 || D < 1 || D > MAXD || E < 1 || B < 1) return 0;
    return fitc_ws_layout(N, Mi, D).per_z * (size_t)B * E * sizeof(double);
}

// adjoint of L = chol(K):  out = sym( Linv' Phi(L' tril(Lbar)) Linv );  Lbar in Pm (destroyed), result in Qm
static int chol_backward(cudaStream_t st, int Zb, int Mi, const double* L, const double* Linv, double* Pm, double* Qm, int ldm, long long zs) {
    const dim3 g2((Mi + 31) / 32, (Mi + 7) / 8, Zb), b2(32, 8);
    tri_op_kernel<<<g2, b2, 0, st>>>(Mi, Pm, ldm, zs, 0);                                     // tril(Lbar)
    int rc = gemm(st, Zb, Mi, Mi, Mi, 1, 0, 1.0, L, ldm, zs, Pm, ldm, zs, 0.0, Qm, ldm, zs);  // L' tril(Lbar)
    if (rc) return rc;
    tri_op_kernel<<<g2, b2, 0, st>>>(Mi, Qm, ldm, zs, 1);                                     // Phi
    rc = gemm(st, Zb, Mi, Mi, Mi, 1, 0, 1.0, Linv, ldm, zs, Qm, ldm, zs, 0.0, Pm, ldm, zs);   // Linv' P
    if (rc) return rc;
    rc = gemm(st, Zb, Mi, Mi, Mi, 0, 0, 1.0, Pm, ldm, zs, Linv, ldm, zs, 0.0, Qm, ldm, zs);   // ... Linv
    if (rc) return rc;
    tri_op_kernel<<<g2, b2, 0, st>>>(Mi, Qm, ldm, zs, 2);                                     // sym
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

int pilco_fitc_nlml(int N, int Mi, int D, int E, int B,
                    const double* X, const double* Y,                 /* [N,D], [N,E] shared by the batch */
                    const double* Z,                                  /* [B,E,Mi,D] */
                    const double* ell, const double* sf2, const double* sn2,   /* [B,E,D], [B,E], [B,E] */
                    double* nlml, double* g_ell, double* g_sf2, double* g_sn2, double* g_Z, int* info,
                    void* ws, size_t ws_bytes, pilco_stream_t stream) {
    if (!X || !Y || !Z || !ell || !sf2 || !sn2 || !nlml || !g_ell || !g_sf2 || !g_sn2 || !g_Z || !ws) return PILCO_ERR_NULL;
    if (N < 1 || Mi < 1 || D < 1 || D > MAXD || E < 1 || E > MAXE || B < 1) return PILCO_ERR_DIM;
    if (ws_bytes < pilco_fitc_nlml_workspace_bytes(N, Mi, D, E, B)) return PILCO_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int Zb = B * E, ldm = pad64(Mi), ldn = pad64(N);
    const FitcWs W = fitc_ws_layout(N, Mi, D);
    const long long zs = (long long)W.per_z;                           // every array is addressed base + z*zs
    double* w = (double*)ws;
    if (info) cudaMemsetAsync(info, 0, sizeof(int) * B, st);
    cudaMemsetAsync(ws, 0, W.per_z * (size_t)Zb * sizeof(double), st);
    // Gram blocks; per (b,e) inducing inputs: the batch index of gram_kernel runs over z with E' = 1
    GramArgs guu{Mi, Mi, D, 1, Z, (long long)Mi * D, Z, (long long)Mi * D, ell, D, sf2, 1, nullptr, 0, 0.0, w + W.Kuu0, ldm, zs, Mi, Mi, 0};
    launch_hi(gram_kernel, dim3((Mi + 31) / 32, (Mi + 7) / 8, Zb), dim3(32, 8), 0, st, guu);
    GramArgs gul{Mi, Mi, D, 1, Z, (long long)Mi * D, Z, (long long)Mi * D, ell, D, sf2, 1, nullptr, 0, 1e-6, w + W.Luu, ldm, zs, Mi, Mi, 0};
    launch_hi(gram_kernel, dim3((Mi + 31) / 32, (Mi + 7) / 8, Zb), dim3(32, 8), 0, st, gul);
    GramArgs guf{Mi, N, D, 1, Z, (long long)Mi * D, X, 0, ell, D, sf2, 1, nullptr, 0, 0.0, w + W.Kuf, ldn, zs, Mi, N, 0};
    launch_hi(gram_kernel, dim3((N + 31) / 32, (Mi + 7) / 8, Zb), dim3(32, 8), 0, st, guf);
    CUDA_LAUNCH_CHECK();
    { int rcc = chol_launch(st, Zb, Mi, w + W.Luu, ldm, zs, E, info); if (rcc) return rcc; }
    tri_op_kernel<<<dim3((Mi + 31) / 32, (Mi + 7) / 8, Zb), dim3(32, 8), 0, st>>>(Mi, w + W.Luu, ldm, zs, 0);     // strict upper := 0
    CUDA_LAUNCH_CHECK();
    int rc = tri_inverse(st, Zb, Mi, w + W.Luu, ldm, zs, w + W.LinvU, ldm, zs, w + W.Ts, zs);
    if (rc) return rc;
    rc = gemm(st, Zb, Mi, N, Mi, 0, 0, 1.0, w + W.LinvU, ldm, zs, w + W.Kuf, ldn, zs, 0.0, w + W.V, ldn, zs);        // V
    if (rc) return rc;
    fitc_nu_kernel<<<dim3((N + 127) / 128, Zb), 128, 0, st>>>(Mi, N, E, w + W.V, ldn, zs, Y, sf2, sn2, w + W.T1, w + W.nu, w + W.ynu);
    CUDA_LAUNCH_CHECK();
    rc = gemm(st, Zb, Mi, Mi, N, 0, 1, 1.0, w + W.T1, ldn, zs, w + W.V, ldn, zs, 0.0, w + W.Bm, ldm, zs);            // V diag(1/nu) V'
    if (rc) return rc;
    add_diag_const_kernel<<<dim3((Mi + 127) / 128, Zb), 128, 0, st>>>(Mi, w + W.Bm, ldm, zs, 1.0);
    { int rcc = chol_launch(st, Zb, Mi, w + W.Bm, ldm, zs, E, info); if (rcc) return rcc; }                          // L (in Bm)
    tri_op_kernel<<<dim3((Mi + 31) / 32, (Mi + 7) / 8, Zb), dim3(32, 8), 0, st>>>(Mi, w + W.Bm, ldm, zs, 0);
    CUDA_LAUNCH_CHECK();
    rc = tri_inverse(st, Zb, Mi, w + W.Bm, ldm, zs, w + W.LinvB, ldm, zs, w + W.Ts, zs);
    if (rc) return rc;
    matvec_kernel<<<dim3(Mi, Zb), 32, 0, st>>>(Mi, N, 0, w + W.V, ldn, zs, w + W.ynu, zs, 1, w + W.al, zs);          // alpha
    matvec_kernel<<<dim3(Mi, Zb), 32, 0, st>>>(Mi, Mi, 0, w + W.LinvB, ldm, zs, w + W.al, zs, 1, w + W.ga, zs);      // gamma
    matvec_kernel<<<dim3(Mi, Zb), 32, 0, st>>>(Mi, Mi, 1, w + W.LinvB, ldm, zs, w + W.ga, zs, 1, w + W.ab, zs);      // ab = -alpha_bar
    CUDA_LAUNCH_CHECK();
    // Bbar = chol_backward(L, Lbar)
    fitc_lbar_kernel<<<dim3((Mi + 31) / 32, (Mi + 7) / 8, Zb), dim3(32, 8), 0, st>>>(Mi, w + W.Bm, ldm, zs, w + W.ab, w + W.ga, w + W.Pm);
    rc = chol_backward(st, Zb, Mi, w + W.Bm, w + W.LinvB, w + W.Pm, w + W.Qm, ldm, zs);
    if (rc) return rc;
    rc = gemm(st, Zb, Mi, N, Mi, 0, 0, 1.0, w + W.Qm, ldm, zs, w + W.V, ldn, zs, 0.0, w + W.T1, ldn, zs);           // BV = Bbar V
    if (rc) return rc;
    fitc_cols_bwd_kernel<<<dim3((N + 127) / 128, Zb), 128, 0, st>>>(Mi, N, E, w + W.V, w + W.T1, ldn, zs, Y, w + W.nu, w + W.ynu, w + W.ab, w + W.nub);
    CUDA_LAUNCH_CHECK();
    rc = gemm(st, Zb, Mi, N, Mi, 1, 0, 1.0, w + W.LinvU, ldm, zs, w + W.T1, ldn, zs, 0.0, w + W.T2, ldn, zs);        // Kuf_bar = Luu^-T Vbar
    if (rc) return rc;
    rc = gemm(st, Zb, Mi, Mi, N, 0, 1, -1.0, w + W.T2, ldn, zs, w + W.V, ldn, zs, 0.0, w + W.Pm, ldm, zs);           // Luu_bar = -Kuf_bar V'
    if (rc) return rc;
    rc = chol_backward(st, Zb, Mi, w + W.Luu, w + W.LinvU, w + W.Pm, w + W.Qm, ldm, zs);                           // Kuu_bar
    if (rc) return rc;
    fitc_adjoint_kernel<<<dim3(Mi, Zb), 128, 0, st>>>(Mi, N, D, X, Z, ell, w + W.Kuf, w + W.T2, ldn, w + W.Kuu0, w + W.Qm, ldm, zs,
                                                      w + W.part, g_Z);
    CUDA_LAUNCH_CHECK();
    fitc_final_kernel<<<Zb, 256, 0, st>>>(Mi, N, D, E, Y, ell, sf2, w + W.Bm, ldm, w + W.nu, w + W.nub, w + W.ga, w + W.part, zs,
                                          nlml, g_ell, g_sf2, g_sn2);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

size_t pilco_fitc_workspace_bytes(int N, int Mi, int E) {
    if (N < 1 || Mi < 1 || E < 1) return 0;
    const size_t ldm = pad64(Mi) + 64, ldn = pad64(N);
    // L, Linv, Am, Aminv, iAt, T : E*ldm*ldm each (6) ; Kmn/V, Vg : E*ldm*ldn each (2) ; w, w2 : E*ldm (2)
    return (6 * E * ldm * ldm + 2 * E * ldm * ldn + 2 * E * ldm) * sizeof(double);
}

int pilco_fitc_factorize(int N, int Mi, int D, int E, const double* X, const double* Z, const double* Y,
                         const double* ell, const double* sf2, const double* sn2,
                         double* iK, int ldk, double* beta, int* info, void* ws, size_t ws_bytes,
                         pilco_stream_t stream) {
    if (!X || !Z || !Y || !ell || !sf2 || !sn2 || !iK || !beta || !ws) return PILCO_ERR_NULL;
    if (N < 1 || Mi < 1 || D < 1 || D > MAXD || E < 1 || E > MAXE) return PILCO_ERR_DIM;
    if (ldk < pad64(Mi)) return PILCO_ERR_DIM;
    if (ws_bytes < pilco_fitc_workspace_bytes(N, Mi, E)) return PILCO_ERR_WORKSPACE;
    cudaStream_t st = (cudaStream_t)stream;
    const int ldm = pad64(Mi) + 64, ldn = pad64(N);
    const long long mm = (long long)ldm * ldm, mn = (long long)ldm * ldn;
    double* w0 = (double*)ws;
    double* L = w0;            double* Linv = L + E * mm;   double* Am = Linv + E * mm;
    double* Aminv = Am + E * mm; double* iAt = Aminv + E * mm; double* T = iAt + E * mm;
    double* V = T + E * mm;    double* Vg = V + E * mn;
    double* w = Vg + E * mn;   double* w2 = w + (size_t)E * ldm;
    if (info) cudaMemsetAsync(info, 0, sizeof(int), st);
    cudaMemsetAsync(ws, 0, pilco_fitc_workspace_bytes(N, Mi, E), st);
    // Kmm + 1e-6 I  (smgpr.py:27), Kmn (smgpr.py:28)
    GramArgs gmm{Mi, Mi, D, E, Z, 0, Z, 0, ell, 0, sf2, 0, nullptr, 0, 1e-6, L, ldm, mm, ldm, ldm, 0};
    launch_hi(gram_kernel, dim3((ldm + 31) / 32, (ldm + 7) / 8, E), dim3(32, 8), 0, st, gmm);
    CUDA_LAUNCH_CHECK();
    GramArgs gmn{Mi, N, D, E, Z, 0, X, 0, ell, 0, sf2, 0, nullptr, 0, 0.0, Vg, ldn, mn, Mi, N, 0};
    launch_hi(gram_kernel, dim3((N + 31) / 32, (Mi + 7) / 8, E), dim3(32, 8), 0, st, gmn);     // Kmn -> Vg (temp)
    CUDA_LAUNCH_CHECK();
    { int rcc = chol_launch(st, E, Mi, L, ldm, mm, E, info); if (rcc) return rcc; }                            // L = chol(Kmm)  :29
    CUDA_LAUNCH_CHECK();
    int rc = tri_inverse(st, E, Mi, L, ldm, mm, Linv, ldm, mm, T, mm);                   // Linv = L^-1
    if (rc) return rc;
    rc = gemm(st, E, Mi, N, Mi, 0, 0, 1.0, Linv, ldm, mm, Vg, ldn, mn, 0.0, V, ldn, mn); // V = L^-1 Kmn  :30
    if (rc) return rc;
    fitc_scale_kernel<<<dim3((N + 127) / 128, E), 128, 0, st>>>(Mi, N, V, ldn, mn, Vg, sf2, sn2);   // :31-33
    CUDA_LAUNCH_CHECK();
    rc = gemm(st, E, Mi, Mi, N, 0, 1, 1.0, V, ldn, mn, V, ldn, mn, 0.0, Am, ldm, mm);    // V V^T
    if (rc) return rc;
    add_diag_kernel<<<dim3((Mi + 127) / 128, E), 128, 0, st>>>(Mi, Am, ldm, mm, sn2);    // + sn2 I   :34-35
    CUDA_LAUNCH_CHECK();
    { int rcc = chol_launch(st, E, Mi, Am, ldm, mm, E, info); if (rcc) return rcc; }                           // Am
    CUDA_LAUNCH_CHECK();
    fill(st, T, (size_t)E * mm, 0.0);
    rc = tri_inverse(st, E, Mi, Am, ldm, mm, Aminv, ldm, mm, T, mm);                     // Am^-1
    if (rc) return rc;
    rc = gemm(st, E, Mi, Mi, Mi, 0, 0, 1.0, Aminv, ldm, mm, Linv, ldm, mm, 0.0, iAt, ldm, mm);   // iAt = (L Am)^-1  :36-37
    if (rc) return rc;
    // beta = L^-T Am^-T Am^-1 (V/G) y     (:38-42)
    matvec_kernel<<<dim3(Mi, E), 32, 0, st>>>(Mi, N, 0, Vg, ldn, mn, Y, 1, E, w, ldm);   // w = Vg y_e  (y stride E, offset e)
    CUDA_LAUNCH_CHECK();
    matvec_kernel<<<dim3(Mi, E), 32, 0, st>>>(Mi, Mi, 0, Aminv, ldm, mm, w, ldm, 1, w2, ldm);
    CUDA_LAUNCH_CHECK();
    matvec_kernel<<<dim3(Mi, E), 32, 0, st>>>(Mi, Mi, 1, Aminv, ldm, mm, w2, ldm, 1, w, ldm);
    CUDA_LAUNCH_CHECK();
    matvec_kernel<<<dim3(Mi, E), 32, 0, st>>>(Mi, Mi, 1, Linv, ldm, mm, w, ldm, 1, beta, Mi);
    CUDA_LAUNCH_CHECK();
    // iK = Kmm^-1 - sn2 iAt^T iAt = Linv^T Linv - sn2 iAt^T iAt   (:43-44)
    cudaMemsetAsync(iK, 0, (size_t)E * ldk * ldk * sizeof(double), st);
    rc = gemm(st, E, Mi, Mi, Mi, 1, 0, 1.0, Linv, ldm, mm, Linv, ldm, mm, 0.0, iK, ldk, (long long)ldk * ldk);
    if (rc) return rc;
    // iK -= sn2[e] * iAt^T iAt
    rc = gemm(st, E, Mi, Mi, Mi, 1, 0, 1.0, iAt, ldm, mm, iAt, ldm, mm, 0.0, T, ldm, mm);
    if (rc) return rc;
    fitc_axpy_kernel<<<dim3((Mi + 31) / 32, (Mi + 7) / 8, E), dim3(32, 8), 0, st>>>(Mi, iK, ldk, (long long)ldk * ldk, T, ldm, mm, sn2);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

}  // extern "C"

// ---- full-covariance branch of pilco_gp_predict (gp_predict.cu) ----------------------------------------------------
// GPR.predict_f / GPRFITC.predict_f with full_cov=True:  cov_e = K_e(Xs, Xs) - W K*',  W = K* iK_e,  K* = K_e(Xs, centres).
// K* and W [E, B, pad64(n)] live in ws (the output is O(B^2) already); arguments validated by the caller.
int gp_predict_full_cov(const pilco_gp_model* gp, int B, const double* Xs, double* cov, double* ws, cudaStream_t st) {
    const int n = gp->n, D = gp->D, E = gp->E, ldn = pad64(n);
    const long long ms = (long long)B * ldn, cs = (long long)B * B, ks = (long long)gp->ldk * gp->ldk;
    double* Ks = ws;
    double* W = Ks + (size_t)E * ms;
    GramArgs gk{B, n, D, E, Xs, 0, gp->X, 0, gp->ell, 0, gp->sf2, 0, nullptr, 0, 0.0, Ks, ldn, ms, B, ldn, 0};
    launch_pri(false, gram_kernel, dim3((ldn + 31) / 32, (B + 7) / 8, E), dim3(32, 8), 0, st, gk);
    GramArgs gc{B, B, D, E, Xs, 0, Xs, 0, gp->ell, 0, gp->sf2, 0, nullptr, 0, 0.0, cov, B, cs, B, B, 0};
    launch_pri(false, gram_kernel, dim3((B + 31) / 32, (B + 7) / 8, E), dim3(32, 8), 0, st, gc);
    CUDA_LAUNCH_CHECK();
    int rc = gemm(st, E, B, n, n, 0, 0, 1.0, Ks, ldn, ms, gp->iK, gp->ldk, ks, 0.0, W, ldn, ms);          // W = K* iK
    if (rc) return rc;
    rc = gemm(st, E, B, B, n, 0, 1, -1.0, W, ldn, ms, Ks, ldn, ms, 1.0, cov, B, cs);                        // cov -= W K*'
    if (rc) return rc;
    // W K*' is symmetric only up to round-off growing with cond(iK): average the two triangles (GPflow's K** - A'A is exact)
    tri_op_kernel<<<dim3((B + 31) / 32, (B + 7) / 8, E), dim3(32, 8), 0, st>>>(B, cov, B, cs, 2);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}
