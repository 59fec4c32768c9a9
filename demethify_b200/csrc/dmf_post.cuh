// dmf_post.cuh — the steps right before and right after the deconvolution path that used to be host / library code
// (SURVEY.md 8 f4):
//   nndsvd_split_kernel    sign split, norms and scaling of NNDSVD (init_func.py:46-69) on the singular vectors of a thin SVD
//   percentile_kernel      lower / upper percentile over the B bootstrap resamples of every entry (np.percentile, linear rule;
//                          bootstrap.py:53-54, :77-78) by selection - no sort of the B x P stack
//   labels_kernel / consensus_kernel   consensus matrix of the restarts' argmax labels (ic.py:24-37)
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace dmf {

// ------------------------------------------------------------------------------------------------
// One CTA per component i.  U is M x ldu (row-major, column i is the i-th left singular vector), Vh is r x ldv (row i the i-th
// right singular vector).  W is M x rank, H is rank x N (both row-major, fully written).
// Component 0: sqrt(S_0) |u_0|, sqrt(S_0) |v_0|.  Component i >= 1: the sign pattern (positive or negative parts of u_i, v_i)
// with the larger product of norms, scaled by sqrt(S_i * term) / norm.  Entries below 1e-11 become 0.
static __global__ void __launch_bounds__(256) nndsvd_split_kernel(const double* __restrict__ U, long long ldu, const double* __restrict__ S,
                                                                  const double* __restrict__ Vh, long long ldv, long long M, int N, int rank,
                                                                  double* __restrict__ W, double* __restrict__ H) {
    __shared__ double red[4][8];
    __shared__ double tot[4];
    const int i = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    double s[4] = {0.0, 0.0, 0.0, 0.0};      // |u+|^2, |u-|^2, |v+|^2, |v-|^2 (fixed order: thread stride, warp tree, warps in order)
    if (i > 0) {
        for (long long m = tid; m < M; m += blockDim.x) {
            const double v = U[m * ldu + i];
            const double p = fmax(v, 0.0), n = fmax(-v, 0.0);
            s[0] = fma(p, p, s[0]);
            s[1] = fma(n, n, s[1]);
        }
        for (int j = tid; j < N; j += blockDim.x) {
            const double v = Vh[(long long)i * ldv + j];
            const double p = fmax(v, 0.0), n = fmax(-v, 0.0);
            s[2] = fma(p, p, s[2]);
            s[3] = fma(n, n, s[3]);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
            if (lane == 0) red[k][warp] = s[k];
        }
        __syncthreads();
        if (tid < 4) {
            double t = 0.0;
            for (int w = 0; w < 8; ++w) t += red[tid][w];
            tot[tid] = t;
        }
        __syncthreads();
    }
    double fu, fv;
    bool positive = true;
    if (i == 0) {
        fu = fv = sqrt(S[0]);
    } else {
        const double n_up = sqrt(tot[0]), n_un = sqrt(tot[1]), n_vp = sqrt(tot[2]), n_vn = sqrt(tot[3]);
        const double termp = n_up * n_vp, termn = n_un * n_vn;
        positive = termp >= termn;
        const double term = positive ? termp : termn;
        fu = sqrt(S[i] * term) / (positive ? n_up : n_un);
        fv = sqrt(S[i] * term) / (positive ? n_vp : n_vn);
    }
    for (long long m = tid; m < M; m += blockDim.x) {
        const double v = U[m * ldu + i];
        double w = i == 0 ? fu * fabs(v) : fu * (positive ? fmax(v, 0.0) : fmax(-v, 0.0));
        if (w < 1e-11) w = 0.0;
        W[m * rank + i] = w;
    }
    for (int j = tid; j < N; j += blockDim.x) {
        const double v = Vh[(long long)i * ldv + j];
        double h = i == 0 ? fv * fabs(v) : fv * (positive ? fmax(v, 0.0) : fmax(-v, 0.0));
        if (h < 1e-11) h = 0.0;
        H[(long long)i * N + j] = h;
    }
}

// ------------------------------------------------------------------------------------------------
// np.percentile(stack, [q_lo, q_hi], axis=0) with the default linear rule: virtual index (B - 1) q / 100, value
// a + (b - a) g for g < 0.5, b - (b - a)(1 - g) otherwise (numpy's _lerp).  One thread per entry p; stack is B x P row-major, so
// the threads of a warp read consecutive addresses for every b.  The thread keeps the KS smallest and the KL largest values seen
// so far in two sorted arrays (insertion): KS = floor((B-1) q_lo/100) + 2, KL = B - floor((B-1) q_hi/100), both <= KMAX.
// A NaN among the B values makes both outputs NaN, as np.percentile does (it sorts NaN last and then returns np.nan); the
// comparisons of the insertion would otherwise skip it, or keep it and block every later insertion.
template <int KMAX>
__global__ void __launch_bounds__(128) percentile_kernel(const double* __restrict__ stack, int B, long long P, double q_lo, double q_hi,
                                                         double* __restrict__ out_lo, double* __restrict__ out_hi) {
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    const double vlo = (double)(B - 1) * (q_lo / 100.0), vhi = (double)(B - 1) * (q_hi / 100.0);
    const int klo = (int)floor(vlo), khi = (int)floor(vhi);
    const double glo = vlo - (double)klo, ghi = vhi - (double)khi;
    const int KS = min(klo + 2, B), KL = min(B - khi, B);
    double sm[KMAX], lg[KMAX];         // sm ascending (the KS smallest), lg descending (the KL largest)
    int ns = 0, nl = 0;
    bool nan = false;
    for (int b = 0; b < B; ++b) {
        const double v = stack[(long long)b * P + p];
        if (v != v) { nan = true; continue; }
        if (ns < KS || v < sm[ns - 1]) {
            int k = ns < KS ? ns++ : ns - 1;
            while (k > 0 && sm[k - 1] > v) { sm[k] = sm[k - 1]; --k; }
            sm[k] = v;
        }
        if (nl < KL || v > lg[nl - 1]) {
            int k = nl < KL ? nl++ : nl - 1;
            while (k > 0 && lg[k - 1] < v) { lg[k] = lg[k - 1]; --k; }
            lg[k] = v;
        }
    }
    if (nan) {
        out_lo[p] = out_hi[p] = __longlong_as_double(0x7ff8000000000000ll);     // np.nan
        return;
    }
    auto lerp = [](double a, double b, double g) { const double d = b - a; return g >= 0.5 ? b - d * (1.0 - g) : a + d * g; };
    {
        const double a = sm[min(klo, B - 1)], b = sm[min(klo + 1, B - 1)];
        out_lo[p] = lerp(a, b, glo);
    }
    {
        // sorted ascending: a[khi] is the (B - khi)-th largest = lg[B - khi - 1], a[khi + 1] = lg[B - khi - 2]
        const double a = lg[B - khi - 1], b = lg[max(B - khi - 2, 0)];
        out_hi[p] = lerp(a, khi + 1 <= B - 1 ? b : a, ghi);
    }
}

// ------------------------------------------------------------------------------------------------
// ic.py:24-37: labels[r][j] = argmax_k alpha_r[k][j] (first maximum, np.argmax: a NaN counts as the maximum, the first one wins), consensus[i][j] = mean_r (labels[r][i] == labels[r][j])
static __global__ void labels_kernel(const double* __restrict__ alpha, int n_runs, int Kt, int N, int* __restrict__ labels) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n_runs * N) return;
    const int r = e / N, j = e - r * N;
    const double* a = alpha + (size_t)r * Kt * N + j;
    int best = 0;
    double bv = a[0];
    for (int k = 1; k < Kt; ++k) {
        const double v = a[(size_t)k * N];
        if (v > bv || (v != v && bv == bv)) { bv = v; best = k; }
    }
    labels[e] = best;
}
static __global__ void consensus_kernel(const int* __restrict__ labels, int n_runs, int N, double* __restrict__ consensus) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (long long)N * N) return;
    const int i = (int)(e / N), j = (int)(e - (long long)i * N);
    double s = 0.0;
    for (int r = 0; r < n_runs; ++r) s += (labels[(size_t)r * N + i] == labels[(size_t)r * N + j]) ? 1.0 : 0.0;
    consensus[e] = s / (double)n_runs;
}

}  // namespace dmf
