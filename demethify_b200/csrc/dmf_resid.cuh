// dmf_resid.cuh — the row reductions of the NNDSVD initialisation (init_func.py:17-93) when the CpG rows are sharded over GPUs.
// The thin SVD of the M x N residual is replaced by the eigen-decomposition of its N x N Gram matrix; every quantity that sums
// over rows is published per GPU so that the caller can all-reduce it:
//   resid_gram_kernel     G = sum_m r_m r_m^T  (N x N)
//   resid_project_kernel  U = r Vh^T diag(1 / sigma) for the GPU's rows and the per-component sums |u+|^2, |u-|^2
//   nndsvd_apply_kernel   W rows and H from U and the all-reduced sums, with the rule of nndsvd_split_kernel
// r_mj = max(x_mj - R_m . H1_.j, 1e-8) (K > 0: the floored residual of the partial / purity SVD init, init_func.py:23-24) or
// r_mj = x_mj (K = 0: nndsvd_initialize on X).  The residual is formed on the fly and never stored in global memory.
#pragma once
#include "dmf_fused.cuh"     // dmma884

namespace dmf {

constexpr int kGramTile = 64;                       // G is produced in 64 x 64 tiles of its upper triangle, one grid row per tile
constexpr int kResPitch = 2 * kGramTile + 4;        // doubles per residual row in shared memory (the tile's two column blocks)
constexpr int kResMaxRows = 32;                     // row-tile bound of resid_gram_kernel (multiple of the MMA k = 4)
constexpr int kMaxResidN = 2 * kConsumers;          // N supported: the library's limit

struct ResidArgs {
    Geom g;                 // row tiles of X (source 0) and R_trunc (source 2); g.N, g.K; n_parts CTAs split the rows of a G tile
    const FitDev* fits;     // one descriptor per G tile (blockIdx.y): X, Rk and the tile's part / gpart / tickets
    const double* H1;       // K x N
    double* G;              // N x N
    int* neg;               // K = 0: set to 1 when a negative entry of X is seen
    int nt;                 // 64-column blocks, ceil(N / 64)
};

// tile t of the upper triangle, row by row: (0,0) (0,1) .. (0,nt-1) (1,1) ..
__device__ __forceinline__ void tri_tile(int t, int nt, int& bi, int& bj) {
    bi = 0;
    while (t >= nt - bi) { t -= nt - bi; ++bi; }
    bj = bi + t;
}

// One CTA = one 64 x 64 tile of G over a share of the row tiles.  Per row tile: the 256 threads form the residual of the tile's
// (up to) 128 columns in shared memory (thread = column, K fused multiply-adds with the H1 column held in registers), then warp w
// accumulates rows 8w .. 8w+7 of the G tile on the FP64 tensor cores (mma.m8n8k4: 4 CpG rows per MMA, the residual rows on
// the K side).  Per-CTA tiles are summed by hier_reduce in a fixed order: bit-reproducible for a given grid.
__global__ void __launch_bounds__(kThreads, 1) resid_gram_kernel(const ResidArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    const Geom& g = a.g;
    const FitDev f = a.fits[blockIdx.y];
    CtaCtx c;
    cta_setup(g, smem, c);
    unsigned char* stages = smem + kCtlBytes;
    const uint32_t stages32 = smem_u32(stages);
    const size_t ring_bytes = (size_t)n_stages(g) * g.stage_bytes;
    double* res = reinterpret_cast<double*>(stages + (ring_bytes > kGramTile * kGramTile * 8 ? ring_bytes : kGramTile * kGramTile * 8));
    int bi, bj;
    tri_tile((int)blockIdx.y, a.nt, bi, bj);
    const bool diag = bi == bj;
    const int ncols = diag ? kGramTile : 2 * kGramTile;
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(double), g.offX, 0, 0, 0};
        src[1] = {nullptr, 0, 0, 0, 0, 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(double), g.offR, 0, 0, 0};
    }
    // the column this thread forms: slot cs of the tile's [bi block | bj block], rows rp, rp + rstride, ...
    const int cs = threadIdx.x % ncols, rp = threadIdx.x / ncols, rstride = kThreads / ncols;
    const int gc = cs < kGramTile ? bi * kGramTile + cs : bj * kGramTile + cs - kGramTile;
    const bool valid = gc < g.N;
    double h[kMaxKt];
#pragma unroll
    for (int k = 0; k < kMaxKt; ++k) h[k] = (valid && k < g.K) ? a.H1[(size_t)k * g.N + gc] : 0.0;
    bool neg = false;
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, 3);
    const int w = c.warp, lane = c.lane;
    const int coff = diag ? 0 : kGramTile;
    double acc[8][2];
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) acc[nb][0] = acc[nb][1] = 0.0;
    for (; cr.it < c.n_my; cr.advance(g, stages32)) {
        produce_next(g, f, c, pr, stages32, 3);
        mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
        const uint32_t sb = cr.sb;
        const int nrows = cr.rows(g, c);
        for (int r = rp; r < g.tile_rows; r += rstride) {
            double v = 0.0;                               // rows past the end of the matrix contribute nothing
            if (valid && r < nrows) {
                double x;
                lds1(sb + g.offX + (uint32_t)((r * g.ldx + gc) * sizeof(double)), x);
                if (g.K) {
                    double s = 0.0;
#pragma unroll
                    for (int k = 0; k < kMaxKt; ++k)
                        if (k < g.K) {
                            double rk;
                            lds1(sb + g.offR + (uint32_t)((r * g.ldr + k) * sizeof(double)), rk);
                            s = fma(rk, h[k], s);
                        }
                    v = fmax(x - s, 1e-8);
                } else {
                    v = x;
                    neg |= x < 0.0;
                }
            }
            res[r * kResPitch + cs] = v;
        }
        __syncwarp();
        if (lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));     // the stage is no longer read: the residual is in `res`
        __syncthreads();
        // A (8 x 4) = rows 8w .. 8w+7 of the tile against 4 CpG rows, B (4 x 8) = the same CpG rows against column block nb
        for (int k0 = 0; k0 < g.tile_rows; k0 += 4) {
            const double* rrow = res + (k0 + (lane & 3)) * kResPitch;
            const double av = rrow[w * 8 + (lane >> 2)];
#pragma unroll
            for (int nb = 0; nb < 8; ++nb) dmma884(acc[nb][0], acc[nb][1], av, rrow[coff + nb * 8 + (lane >> 2)]);
        }
        __syncthreads();                                  // `res` is rewritten by the next tile
    }
    if (neg) atomicOr(a.neg, 1);
    constexpr int TT = kGramTile * kGramTile;
    double* part = f.part + (size_t)part_id(g) * g.part_stride;
    const int row = w * 8 + (lane >> 2);
#pragma unroll
    for (int nb = 0; nb < 8; ++nb) {
        part[row * kGramTile + nb * 8 + 2 * (lane & 3)] = acc[nb][0];
        part[row * kGramTile + nb * 8 + 2 * (lane & 3) + 1] = acc[nb][1];
    }
    double* tot = reinterpret_cast<double*>(stages);
    if (!hier_reduce(g, f, tot, TT, &c.ctl->flag)) return;
    for (int e = threadIdx.x; e < TT; e += blockDim.x) {
        const int i = bi * kGramTile + e / kGramTile, j = bj * kGramTile + e % kGramTile;
        if (i < g.N && j < g.N && i <= j) {               // the upper triangle, mirrored: G is exactly symmetric
            a.G[(size_t)i * g.N + j] = tot[e];
            a.G[(size_t)j * g.N + i] = tot[e];
        }
    }
}

struct ProjArgs {
    Geom g;                 // M, N, K, ldx, ldr; n_parts CTAs, n_groups, part_stride = 2 rank
    const FitDev* fit;      // part / gpart / tickets of the sums
    const double* X;
    const double* R;
    const double* H1;       // K x N
    const double* Vh;       // rank x N
    const double* inv_s;    // rank
    double* U;              // M x rank
    double* sums;           // 2 rank
    int rank;
};

// One warp per CpG row (rows blockIdx.x * 8 + warp, + 8 gridDim.x, ...): lane l forms r_mj for j = l, l + 32, ... and accumulates
// r_mj Vh[i][j] for every component i; a butterfly gives the row's U entries; lane i keeps the squared positive / negative parts of
// component i over the warp's rows.  Warps, then CTAs (hier_reduce), are summed in a fixed order.
__global__ void __launch_bounds__(kThreads) resid_project_kernel(const ProjArgs a) {
    __shared__ double red[kConsumers / 32][2 * kMaxKt];
    __shared__ double tot[2 * kMaxKt];
    __shared__ int flag;
    const Geom& g = a.g;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double sp = 0.0, sn = 0.0;
    for (long long m = (long long)blockIdx.x * (kThreads / 32) + w; m < g.M; m += (long long)gridDim.x * (kThreads / 32)) {
        double acc[kMaxKt];
#pragma unroll
        for (int i = 0; i < kMaxKt; ++i) acc[i] = 0.0;
        for (int j = lane; j < g.N; j += 32) {
            const double x = a.X[m * g.ldx + j];
            double v = x;
            if (g.K) {
                double s = 0.0;
                for (int k = 0; k < g.K; ++k) s = fma(a.R[m * g.ldr + k], __ldg(&a.H1[(size_t)k * g.N + j]), s);
                v = fmax(x - s, 1e-8);
            }
#pragma unroll
            for (int i = 0; i < kMaxKt; ++i)
                if (i < a.rank) acc[i] = fma(v, __ldg(&a.Vh[(size_t)i * g.N + j]), acc[i]);
        }
        double mine = 0.0;
#pragma unroll
        for (int i = 0; i < kMaxKt; ++i) {
            if (i < a.rank) {
                double t = acc[i];
#pragma unroll
                for (int o = 16; o >= 1; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
                t = __shfl_sync(0xffffffffu, t, 0) * __ldg(&a.inv_s[i]);
                if (lane == i) mine = t;
            }
        }
        if (lane < a.rank) {
            a.U[m * a.rank + lane] = mine;
            const double p = fmax(mine, 0.0), n = fmax(-mine, 0.0);
            sp = fma(p, p, sp);
            sn = fma(n, n, sn);
        }
    }
    if (lane < a.rank) {
        red[w][lane] = sp;
        red[w][a.rank + lane] = sn;
    }
    __syncthreads();
    const FitDev& f = *a.fit;
    double* part = f.part + (size_t)part_id(g) * g.part_stride;
    if (threadIdx.x < 2 * a.rank) {
        double s = 0.0;
        for (int ww = 0; ww < kConsumers / 32; ++ww) s += red[ww][threadIdx.x];
        part[threadIdx.x] = s;
    }
    if (!hier_reduce(g, f, tot, 2 * a.rank, &flag)) return;
    if (threadIdx.x < 2 * a.rank) a.sums[threadIdx.x] = tot[threadIdx.x];
}

// grid (rank, row blocks).  CTA (i, b): the norms of component i of Vh (fixed order, like nndsvd_split_kernel), the sign pattern and
// scale of nndsvd_split_kernel with |u+|, |u-| from `sums`, then W[m][i] for the block's rows and, in block 0, H[i][:].
__global__ void __launch_bounds__(256) nndsvd_apply_kernel(const double* __restrict__ U, long long M, const double* __restrict__ Vh,
                                                           const double* __restrict__ S, const double* __restrict__ sums, int N, int rank,
                                                           double* __restrict__ W, double* __restrict__ H) {
    __shared__ double red[2][8];
    __shared__ double tot[2];
    const int i = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (i > 0) {
        double s[2] = {0.0, 0.0};
        for (int j = tid; j < N; j += blockDim.x) {
            const double v = Vh[(long long)i * N + j];
            const double p = fmax(v, 0.0), n = fmax(-v, 0.0);
            s[0] = fma(p, p, s[0]);
            s[1] = fma(n, n, s[1]);
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
            if (lane == 0) red[k][warp] = s[k];
        }
        __syncthreads();
        if (tid < 2) {
            double t = 0.0;
            for (int ww = 0; ww < 8; ++ww) t += red[tid][ww];
            tot[tid] = t;
        }
        __syncthreads();
    }
    double fu, fv;
    bool positive = true;
    if (i == 0) {
        fu = fv = sqrt(S[0]);
    } else {
        const double n_up = sqrt(sums[i]), n_un = sqrt(sums[rank + i]), n_vp = sqrt(tot[0]), n_vn = sqrt(tot[1]);
        const double termp = n_up * n_vp, termn = n_un * n_vn;
        positive = termp >= termn;
        const double term = positive ? termp : termn;
        fu = sqrt(S[i] * term) / (positive ? n_up : n_un);
        fv = sqrt(S[i] * term) / (positive ? n_vp : n_vn);
    }
    for (long long m = (long long)blockIdx.y * blockDim.x + tid; m < M; m += (long long)gridDim.y * blockDim.x) {
        const double v = U[m * rank + i];
        double wv = i == 0 ? fu * fabs(v) : fu * (positive ? fmax(v, 0.0) : fmax(-v, 0.0));
        if (wv < 1e-11) wv = 0.0;
        W[m * rank + i] = wv;
    }
    if (blockIdx.y == 0)
        for (int j = tid; j < N; j += blockDim.x) {
            const double v = Vh[(long long)i * N + j];
            double hv = i == 0 ? fv * fabs(v) : fv * (positive ? fmax(v, 0.0) : fmax(-v, 0.0));
            if (hv < 1e-11) hv = 0.0;
            H[(long long)i * N + j] = hv;
        }
}

}  // namespace dmf
