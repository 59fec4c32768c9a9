// dmf_wls.cuh — weighted least squares with intercept and non-negativity (init_func.py:8-14, wls_intercept):
//   min_{c >= 0, b}  sum_m d_m (y_m - R_m c - b)^2 ,   result c / max(sum c, 1e-10)
// for every sample column at once.  sklearn's LinearRegression(positive=True, fit_intercept=True) centres R and y
// with the weights and hands sqrt(d)-scaled data to scipy.optimize.nnls; here ONE streaming pass accumulates the
// weighted moment matrix  Z_j = sum_m d_mj z z^T,  z = [1, y_mj, R_m0 .. R_m,K-1]  per sample j (fp64, fixed
// order), and a second tiny kernel centres it and runs Lawson-Hanson on the K x K normal equations per sample.
#pragma once
#include "dmf_kernels.cuh"

namespace dmf {

constexpr int kWlsBlock = 8;   // the moment matrix is produced in 8 x 8 blocks (bi <= bj), one launch per block pair

struct WlsArgs {
    Geom g;                 // K = columns of R_full (known + optional U), nu = 0 semantics handled via ldu/nup
    const FitDev* fits;     // one descriptor: X, D, Rk, U (optional second block of R_full), part/gpart/tickets
    double* mom;            // [(Kz) x (Kz)][N] moment matrix, Kz = Kfull + 2
    int Kfull;              // total regressors (K + n_u)
    int bi, bj;             // block pair of this launch
    int y_is_dx;            // 1: y = d * x (demethify.py:212), 0: y = x
};

// z value idx of a row: 0 -> 1, 1 -> y, 2.. -> regressors
template <typename T>
__device__ __forceinline__ double wls_z(const WlsArgs& a, uint32_t sb, int r, int idx, double y) {
    const Geom& g = a.g;
    if (idx == 0) return 1.0;
    if (idx == 1) return y;
    const int k = idx - 2;
    if (k >= a.Kfull) return 0.0;
    T v;
    if (k < g.K) lds1(sb + g.offR + (uint32_t)((r * g.ldr + k) * sizeof(T)), v);
    else lds1(sb + g.offU + (uint32_t)((r * g.ldu + (k - g.K)) * sizeof(T)), v);
    return (double)v;
}

template <typename T, typename WT>
__global__ void __launch_bounds__(kThreads, 1) wls_moments_kernel(const WlsArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const Geom& g = a.g;
    const FitDev f = a.fits[0];
    CtaCtx c;
    cta_setup(g, smem, c);
    unsigned char* stages = smem + kCtlBytes;
    const uint32_t stages32 = smem_u32(stages);
    constexpr int NSRC = 4;
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(T), g.offX, 1, 0, 0};
        src[1] = {f.D, g.ldd * (long long)sizeof(WT), g.offD, 1, 0, 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(T), g.offR, 1, 0, 0};
        src[3] = {g.nu ? f.U : nullptr, g.ldu * (long long)sizeof(T), g.offU, 0, 0, 0};
    }
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, NSRC);
    const int tc = c.ctid % g.ntc, gr = c.ctid / g.ntc;
    const bool colvalid = tc < g.N;
    const int j = colvalid ? tc : 0;
    double acc[kWlsBlock][kWlsBlock];
#pragma unroll
    for (int p = 0; p < kWlsBlock; ++p)
#pragma unroll
        for (int q = 0; q < kWlsBlock; ++q) acc[p][q] = 0.0;
    for (; cr.it < c.n_my; cr.advance(g, stages32)) {
        produce_next(g, f, c, pr, stages32, NSRC);
        mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
        const uint32_t sb = cr.sb;
        const int nrows = cr.rows(g, c);
        if (colvalid) {
            for (int r = gr; r < nrows; r += g.rg) {
                T xv[1], dv[1];
                ldsC<T, 1>(sb + g.offX + (uint32_t)((r * g.ldx + j) * sizeof(T)), xv);
                WLoad<T, WT, 1>::ld(sb + g.offD + (uint32_t)((r * g.ldd + j) * sizeof(WT)), dv);
                const double d = (double)dv[0];
                const double y = a.y_is_dx ? d * (double)xv[0] : (double)xv[0];
                double za[kWlsBlock], zb[kWlsBlock];
#pragma unroll
                for (int p = 0; p < kWlsBlock; ++p) {
                    za[p] = wls_z<T>(a, sb, r, a.bi * kWlsBlock + p, y);
                    zb[p] = (a.bi == a.bj) ? za[p] : wls_z<T>(a, sb, r, a.bj * kWlsBlock + p, y);
                }
#pragma unroll
                for (int p = 0; p < kWlsBlock; ++p) {
                    const double dz = d * za[p];
#pragma unroll
                    for (int q = 0; q < kWlsBlock; ++q) acc[p][q] = fma(dz, zb[q], acc[p][q]);
                }
            }
        }
        __syncwarp();
        if (c.lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));
    }
    __syncthreads();
    // combine the row groups of this CTA in fixed order: scratch[(p*8+q)*N + j]
    double* scratch = reinterpret_cast<double*>(stages);
    const int BN = kWlsBlock * kWlsBlock * g.N;
    for (int gg = 0; gg < g.rg; ++gg) {
        if (gr == gg && colvalid) {
#pragma unroll
            for (int p = 0; p < kWlsBlock; ++p)
#pragma unroll
                for (int q = 0; q < kWlsBlock; ++q) {
                    double* ptr = &scratch[(size_t)(p * kWlsBlock + q) * g.N + j];
                    *ptr = (gg == 0) ? acc[p][q] : (*ptr + acc[p][q]);
                }
        }
        __syncthreads();
    }
    double* part = f.part + (size_t)part_id(g) * g.part_stride;
    for (int e = threadIdx.x; e < BN; e += blockDim.x) part[e] = scratch[e];
    if (!hier_reduce(g, f, scratch, BN, &c.ctl->flag)) return;
    const int Kz = a.Kfull + 2;
    for (int e = threadIdx.x; e < BN; e += blockDim.x) {
        const int pq = e / g.N, jj = e - pq * g.N;
        const int p = a.bi * kWlsBlock + pq / kWlsBlock, q = a.bj * kWlsBlock + pq % kWlsBlock;
        // a diagonal block accumulates both (p, q) and (q, p), which round differently ((d z_p) z_q vs (d z_q) z_p): only the
        // upper entry is stored, mirrored, so that each moment has one writer and the matrix is exactly symmetric
        if (p < Kz && q < Kz && p <= q) {
            a.mom[((size_t)p * Kz + q) * g.N + jj] = scratch[e];
            a.mom[((size_t)q * Kz + p) * g.N + jj] = scratch[e];
        }
    }
}

#ifndef DMF_INST_BODY     // launched by dmf_api.cu only: the instantiation units leave this kernel out
// Lawson-Hanson active-set NNLS on the centred normal equations, one thread per sample.
// Third-party algorithm on the reference path: scipy.optimize.nnls (reached through sklearn, init_func.py:9).
static __global__ void wls_nnls_kernel(const double* __restrict__ mom, int K, int N, long long M, double* __restrict__ out /* [K][ldo] */,
                                       long long ldo, int* __restrict__ status) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= N) return;
    const int Kz = K + 2;
    auto Z = [&](int p, int q) { return mom[((size_t)p * Kz + q) * N + j]; };
    double G[kMaxKt][kMaxKt], b[kMaxKt], x[kMaxKt], s[kMaxKt], w[kMaxKt], L[kMaxKt][kMaxKt];
    bool pas[kMaxKt];
    const double sw = Z(0, 0);
    const double ybar = Z(0, 1) / sw;
    for (int p = 0; p < K; ++p) {
        const double rp = Z(0, 2 + p) / sw;
        b[p] = Z(1, 2 + p) - rp * Z(0, 1);                       // sum d (R_p - rbar_p)(y - ybar)
        for (int q = 0; q < K; ++q) G[p][q] = Z(2 + p, 2 + q) - rp * Z(0, 2 + q);
        x[p] = 0.0; pas[p] = false;
    }
    (void)ybar;
    double nb = 0.0;
    for (int p = 0; p < K; ++p) nb += fabs(b[p]);
    const double tolx = 10.0 * (double)(M > K ? M : K) * 2.220446049250313e-16;     // threshold on the coefficients: unscaled
    const double tol = tolx * nb;                                                     // threshold on the dual w = A^T (b - A x): scaled by |A^T b|_1
    bool singular = false;
    // solve G_PP s_P = b_P by Cholesky on the passive set
    auto solve = [&]() {
        int idx[kMaxKt], n = 0;
        for (int p = 0; p < K; ++p) { s[p] = 0.0; if (pas[p]) idx[n++] = p; }
        for (int i = 0; i < n; ++i)
            for (int k = 0; k <= i; ++k) {
                double v = G[idx[i]][idx[k]];
                for (int t = 0; t < k; ++t) v -= L[i][t] * L[k][t];
                if (i == k && !(v > 0.0)) singular = true;       // collinear regressors on the passive set
                L[i][k] = (i == k) ? sqrt(v > 0.0 ? v : 1e-300) : v / L[k][k];
            }
        double y[kMaxKt];
        for (int i = 0; i < n; ++i) {
            double v = b[idx[i]];
            for (int t = 0; t < i; ++t) v -= L[i][t] * y[t];
            y[i] = v / L[i][i];
        }
        for (int i = n - 1; i >= 0; --i) {
            double v = y[i];
            for (int t = i + 1; t < n; ++t) v -= L[t][i] * s[idx[t]];
            s[idx[i]] = v / L[i][i];
        }
    };
    auto grad = [&]() {
        for (int p = 0; p < K; ++p) {
            double v = b[p];
            for (int q = 0; q < K; ++q) v -= G[p][q] * x[q];
            w[p] = v;
        }
    };
    grad();
    int it = 0;
    const int max_it = 3 * K;
    while (true) {
        int best = -1;
        double wb = tol;
        for (int p = 0; p < K; ++p)
            if (!pas[p] && w[p] > wb) { wb = w[p]; best = p; }
        if (best < 0) break;
        pas[best] = true;
        solve();
        while (it < max_it) {
            double smin = 1e300;
            for (int p = 0; p < K; ++p)
                if (pas[p] && s[p] < smin) smin = s[p];
            if (smin > 0.0) break;
            ++it;
            double step = 1e300;
            for (int p = 0; p < K; ++p)
                if (pas[p] && s[p] <= 0.0) { const double t = x[p] / (x[p] - s[p]); if (t < step) step = t; }
            for (int p = 0; p < K; ++p) x[p] = x[p] * (1.0 - step) + step * s[p];
            for (int p = 0; p < K; ++p)
                if (x[p] <= tolx) { pas[p] = false; }
            for (int p = 0; p < K; ++p)
                if (!pas[p]) x[p] = 0.0;
            solve();
        }
        for (int p = 0; p < K; ++p) x[p] = s[p];
        grad();
    }
    double sum = 0.0;
    for (int p = 0; p < K; ++p) sum += x[p];
    const double den = sum > 1e-10 ? sum : 1e-10;
    for (int p = 0; p < K; ++p) out[(size_t)p * ldo + j] = x[p] / den;
    if (!(sum == sum)) atomicOr(status, 1);           // NaN proportions (e.g. a sample whose weights are all zero)
    if (singular) atomicOr(status, 2);
}
#endif  // DMF_INST_BODY

}  // namespace dmf
