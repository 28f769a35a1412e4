// gp_predict.cu -- GP predictive at deterministic test inputs (fp64):
//   pilco_gp_predict   gpflow.models.GPR.predict_f / GPRFITC.predict_f on the per-output models of MGPR / SMGPR
//                      (pilco/models/mgpr.py:28-36, smgpr.py:16-22), and through them predict_y / predict_log_density
//
// From the resident factors of a pilco_gp_model, for every test point x and output e:
//   mean = k*' beta_e,   var = sf2_e - k*' iK_e k*,   k* = k_e(centres, x)
// which is GPflow's predictive exactly, for the exact GP (iK = (K + sn2 I)^-1) and for FITC (iK = Kmm^-1 - sn2 (Kmm A)^-1,
// pilco_fitc_factorize).  iK is the one factor pilco_gp_append keeps up to date as well, so appended models need nothing else.
//
// Diagonal case: ONE fused kernel.  A CTA owns BT test points and one output; it writes the SE-ARD cross-Gram row block
// K*[BT, n] into shared memory (table exp of exp_table.cuh), forms the mean as a warp dot product with beta, and the
// quadratic form rowsum((K* iK) o K*) with DMMA.8x8x4: warps take 8-column slices of W = K* iK (iK fragments read from
// L2), multiply them into K* in registers and leave per-row partial sums, which are reduced across the 4 lanes of a row
// and then across the 8 warps in a fixed order.  K* never reaches global memory; no workspace; no atomics.  The
// arithmetic of a point depends only on its own row, n and the model, so a point's result is bitwise the same whatever
// the batch size B and its position in the batch.
// Full covariance: gp_predict_full_cov (factorize.cu) with the factorisations' Gram kernel and DMMA GEMM.
#include "common.cuh"

#define GPP_THREADS 256
#define GPP_WARPS (GPP_THREADS / 32)

// row stride of the K* tile: covers round8(n) columns, == 4 (mod 16) doubles so the 8-row x 4-k DMMA A-fragment reads of a
// half-warp hit 16 distinct bank pairs (as GD_LD in factorize.cu)
static inline __host__ __device__ int gpp_ldks(int n) { return ((n + 15) & ~15) + 4; }
static inline size_t gpp_smem_bytes(int n, int bt) {
    return sizeof(double) * ((size_t)EXP_TAB_DOUBLES + (size_t)bt * gpp_ldks(n) + (size_t)bt * MAXD + (size_t)GPP_WARPS * bt);
}
// points per CTA: 32 while the K* tile fits shared memory, then 16, then 8 (n <= 3472).  A function of n only.
static inline int gpp_rows(int n) {
    for (int bt = 32; bt >= 8; bt >>= 1)
        if (gpp_smem_bytes(n, bt) <= PILCO_MAX_SMEM_OPTIN) return bt;
    return 0;
}

struct GppArgs {
    int n, D, E, B;
    const double* X;        // [n,D] centres
    const double* ell;      // [E,D]
    const double* sf2;      // [E]
    const double* beta;     // [E,n]
    const double* iK;       // [E,ldk,ldk] or NULL (mean only)
    int ldk;
    const double* Xs;       // [B,D] test points
    double* mean;           // [B,E] or NULL
    double* var;            // [B,E] or NULL
};

template <int RO>           // row octets per CTA: BT = 8 RO test points
__global__ void __launch_bounds__(GPP_THREADS) gp_predict_kernel(GppArgs a) {
    constexpr int BT = 8 * RO;
    extern __shared__ __align__(16) double gpp_sm[];
    const int n = a.n, D = a.D, E = a.E, ldks = gpp_ldks(n);
    double* tab = gpp_sm;                                   // [EXP_TAB_DOUBLES]
    double* Ks = tab + EXP_TAB_DOUBLES;                     // [BT][ldks]   K*, zero beyond column n
    double* xs = Ks + (size_t)BT * ldks;                    // [BT][MAXD]   test points / ell
    double* red = xs + BT * MAXD;                           // [GPP_WARPS][BT]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int e = blockIdx.y;
    const long long p0 = (long long)blockIdx.x * BT;
    exp_table_init(tab);
    const double* le = a.ell + (size_t)e * D;
    for (int i = tid; i < BT * MAXD; i += GPP_THREADS) {
        const int p = i / MAXD, d = i % MAXD;
        const long long gp = p0 + p;
        xs[i] = (d < D && gp < a.B) ? a.Xs[(size_t)gp * D + d] / le[d] : 0.0;
    }
    __syncthreads();
    // K*[p][j] = sf2 exp(-0.5 |x_p/ell - c_j/ell|^2): thread per centre, its scaled coordinates in registers
    const double sf = a.sf2[e];
    const double* ltab = EXP_LANE_TAB(tab, lane);
    const int ncol = (n + 7) & ~7;
    for (int j = tid; j < ncol; j += GPP_THREADS) {
        if (j >= n) {
#pragma unroll 4
            for (int p = 0; p < BT; ++p) Ks[p * ldks + j] = 0.0;
            continue;
        }
        double cj[MAXD];
#pragma unroll
        for (int d = 0; d < MAXD; ++d) cj[d] = d < D ? a.X[(size_t)j * D + d] / le[d] : 0.0;
#pragma unroll 2
        for (int p = 0; p < BT; ++p) {
            double d2 = 0.0;
#pragma unroll
            for (int d = 0; d < MAXD; ++d) {
                if (d < D) { const double t = xs[p * MAXD + d] - cj[d]; d2 = fma(t, t, d2); }
            }
            Ks[p * ldks + j] = sf * exp_scaled(d2 * (-0.5 * EXP_SC), ltab);
        }
    }
    __syncthreads();
    if (a.mean) {                                           // mean = K* beta_e: warp per point, fixed lane order
        const double* be = a.beta + (size_t)e * n;
        for (int p = warp; p < BT; p += GPP_WARPS) {
            double s = 0.0;
            for (int j = lane; j < n; j += 32) s = fma(Ks[p * ldks + j], be[j], s);
            s = warp_sum(s);
            if (lane == 0 && p0 + p < a.B) a.mean[(size_t)(p0 + p) * E + e] = s;
        }
    }
    if (a.var) {                                            // var = sf2 - rowsum((K* iK) o K*)
        const int g = lane >> 2, t = lane & 3;
        const int kend = (n + 3) & ~3, nco = ncol >> 3;
        const double* iKe = a.iK + (size_t)e * a.ldk * a.ldk;
        double part[RO];
#pragma unroll
        for (int r = 0; r < RO; ++r) part[r] = 0.0;
        for (int co = warp; co < nco; co += GPP_WARPS) {    // 8-column slice c0..c0+7 of W = K* iK
            const int c0 = co * 8;
            double acc[RO][2];
#pragma unroll
            for (int r = 0; r < RO; ++r) acc[r][0] = acc[r][1] = 0.0;
            const double* bp = iKe + (size_t)t * a.ldk + c0 + g;               // B[k = t][col = g] = iK[k0 + t][c0 + g]
            const double* ap = Ks + g * ldks + t;                              // A[row = g][k = t] = K*[8r + g][k0 + t]
#pragma unroll 4
            for (int k0 = 0; k0 < kend; k0 += 4) {
                const double b = __ldg(bp + (size_t)k0 * a.ldk);
#pragma unroll
                for (int r = 0; r < RO; ++r) dmma884(acc[r][0], acc[r][1], ap[r * 8 * ldks + k0], b);
            }
#pragma unroll
            for (int r = 0; r < RO; ++r) {                  // W[row g][cols 2t, 2t+1] * K*[row g][same cols]
                const double* kr = Ks + (r * 8 + g) * ldks + c0 + 2 * t;
                part[r] = fma(acc[r][0], kr[0], part[r]);
                part[r] = fma(acc[r][1], kr[1], part[r]);
            }
        }
#pragma unroll
        for (int r = 0; r < RO; ++r) {
            double v = part[r];
            v += __shfl_xor_sync(0xffffffffu, v, 1);
            v += __shfl_xor_sync(0xffffffffu, v, 2);
            if (t == 0) red[warp * BT + r * 8 + g] = v;
        }
        __syncthreads();
        if (tid < BT && p0 + tid < a.B) {
            double q = 0.0;
#pragma unroll
            for (int w = 0; w < GPP_WARPS; ++w) q += red[w * BT + tid];
            a.var[(size_t)(p0 + tid) * E + e] = sf - q;
        }
    }
}

template <int RO>
static int gpp_launch(const GppArgs& a, cudaStream_t st) {
    const size_t smem = gpp_smem_bytes(a.n, 8 * RO);
    static int attr_done[PILCO_MAX_DEVICES] = {0};
    const int dev = pilco_current_device();
    if (!attr_done[dev]) {
        if (cudaFuncSetAttribute(gp_predict_kernel<RO>, cudaFuncAttributeMaxDynamicSharedMemorySize, PILCO_MAX_SMEM_OPTIN) != cudaSuccess)
            return PILCO_ERR_LAUNCH;
        attr_done[dev] = 1;
    }
    const dim3 grid((unsigned)((a.B + 8 * RO - 1) / (8 * RO)), a.E);
    gp_predict_kernel<RO><<<grid, GPP_THREADS, smem, st>>>(a);
    CUDA_LAUNCH_CHECK();
    return PILCO_OK;
}

// full-covariance branch, factorize.cu (Gram kernel + DMMA GEMM):  cov_e = K_e(Xs, Xs) - (K* iK_e) K*'
int gp_predict_full_cov(const pilco_gp_model* gp, int B, const double* Xs, double* cov, double* ws, cudaStream_t st);

extern "C" {

size_t pilco_gp_predict_workspace_bytes(int n, int D, int E, int B, int full_cov) {
    if (n < 1 || D < 1 || D > MAXD || E < 1 || E > MAXE || B < 0) return 0;
    if (!full_cov) return 0;                                // the fused diagonal kernel needs no scratch
    return (size_t)2 * E * B * pad64(n) * sizeof(double);   // K* and K* iK, [E, B, pad64(n)] each
}

int pilco_gp_predict(const pilco_gp_model* gp, int B, const double* Xs, double* mean, double* var, double* cov,
                     void* ws, size_t ws_bytes, pilco_stream_t stream) {
    if (!gp) return PILCO_ERR_NULL;
    const int n = gp->n, D = gp->D, E = gp->E;
    if (n < 1 || D < 1 || D > MAXD || E < 1 || E > MAXE || (gp->mode != 0 && gp->mode != 1)) return PILCO_ERR_DIM;
    if (gp->X_bs || gp->ell_bs || gp->sf2_bs || gp->beta_bs) return PILCO_ERR_DIM;     // one model, not a batch
    if (B < 0) return PILCO_ERR_DIM;
    if ((var || cov) && !gp->iK) return PILCO_ERR_NULL;                                // variances need iK (mode 0)
    if (gp->iK && gp->ldk < pad64(n)) return PILCO_ERR_DIM;
    if (gpp_rows(n) == 0) return PILCO_ERR_UNSUPPORTED;                                // n beyond the shared-memory K* tile
    if (B == 0) return PILCO_OK;
    if (!gp->X || !gp->ell || !gp->sf2 || !Xs || (mean && !gp->beta)) return PILCO_ERR_NULL;
    if (!mean && !var && !cov) return PILCO_ERR_NULL;
    if (ws_bytes < pilco_gp_predict_workspace_bytes(n, D, E, B, cov != nullptr)) return PILCO_ERR_WORKSPACE;
    if (cov && !ws) return PILCO_ERR_NULL;
    cudaStream_t st = (cudaStream_t)stream;
    if (mean || var) {
        GppArgs a{n, D, E, B, gp->X, gp->ell, gp->sf2, gp->beta, gp->iK, gp->ldk, Xs, mean, var};
        int rc;
        switch (gpp_rows(n)) {
            case 32: rc = gpp_launch<4>(a, st); break;
            case 16: rc = gpp_launch<2>(a, st); break;
            default: rc = gpp_launch<1>(a, st); break;
        }
        if (rc) return rc;
    }
    if (cov) return gp_predict_full_cov(gp, B, Xs, cov, (double*)ws, st);
    return PILCO_OK;
}

}  // extern "C"
