// dmf_kernels.cuh — reference-shaped streaming passes over the tall CpG dimension.
//
// Every kernel is ONE launch = one reference step for all live fits of a batch (grid.y = fit):
//   cost_kernel      : cost_f_w (+ ||R||^2, max d_x at set-up)        deconvolution.py:15-17, 192-204, 218-221
//   u_pass_kernel    : one inner iteration of update_u                deconvolution.py:82-89  (unsup. variant :157-164)
//   alpha_pass_kernel: one inner iteration of update_alpha            deconvolution.py:94-101 + projection :21-37
//                      or one Frank-Wolfe iteration                   deconvolution.py:285-299
//
// Layout: row tiles of X, D, R_trunc, u (and u_prev) are streamed into a shared-memory ring (3 .. 5 stages) with
// 1-D bulk copies (TMA engine, SASS UBLKCP) signalled through mbarriers; the producer duty rotates over the 8 warps,
// every warp computes.  The 256 threads are arranged as (row group g, column thread tc): thread tc owns C adjacent
// sample columns (C = 2: every access is a two-element vector load), keeps its alpha columns in registers and walks
// the rows of the tile.  All row pitches are even and zero padded (ABI contract), so the inner loops are branch free.
// Row-wise sums (U gradient) use a transposed warp-shuffle butterfly, column-wise sums (alpha gradient)
// stay in registers across the whole CTA lifetime; cross-CTA sums go through the deterministic two-level
// reduction of dmf_device.cuh and the LAST CTA applies the step (clip / simplex projection / Frank-Wolfe
// vertex), updates the fit state and re-arms the tickets.
#pragma once
#include "dmf_device.cuh"

namespace dmf {

// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T fma_t(T a, T b, T c);
template <>
__device__ __forceinline__ double fma_t<double>(double a, double b, double c) { return fma(a, b, c); }
template <>
__device__ __forceinline__ float fma_t<float>(float a, float b, float c) { return fmaf(a, b, c); }

// ---- shared-memory loads through 32-bit shared addresses (explicit ld.shared: no 64-bit address math)
__device__ __forceinline__ void lds2(uint32_t addr, double& a, double& b) {
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(a), "=d"(b) : "r"(addr));
}
__device__ __forceinline__ void lds2(uint32_t addr, float& a, float& b) {
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "r"(addr));
}
__device__ __forceinline__ void lds1(uint32_t addr, double& a) { asm volatile("ld.shared.f64 %0, [%1];" : "=d"(a) : "r"(addr)); }
__device__ __forceinline__ void lds1(uint32_t addr, float& a) { asm volatile("ld.shared.f32 %0, [%1];" : "=f"(a) : "r"(addr)); }
// C adjacent elements (C = 1, 2, 4)
template <typename T, int C>
__device__ __forceinline__ void ldsC(uint32_t addr, T (&x)[C]) {
    if (C == 1) lds1(addr, x[0]);
    else {
#pragma unroll
        for (int i = 0; i < C / 2; ++i) lds2(addr + i * 2 * (uint32_t)sizeof(T), x[2 * i], x[(2 * i + 1) % C]);
    }
}
// C adjacent weights, converted to T
template <typename T, typename WT, int C>
struct WLoad {   // WT == T
    static __device__ __forceinline__ void ld(uint32_t addr, T (&d)[C]) { ldsC<T, C>(addr, d); }
};
template <typename T>
struct WLoad<T, uint16_t, 1> {
    static __device__ __forceinline__ void ld(uint32_t addr, T (&d)[1]) {
        uint16_t v;
        asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
        d[0] = (T)v;
    }
};
template <typename T>
struct WLoad<T, uint16_t, 2> {
    static __device__ __forceinline__ void ld(uint32_t addr, T (&d)[2]) {
        uint32_t v;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
        d[0] = (T)(v & 0xffffu);
        d[1] = (T)(v >> 16);
    }
};
template <typename T>
struct WLoad<T, uint16_t, 4> {
    static __device__ __forceinline__ void ld(uint32_t addr, T (&d)[4]) {
        uint32_t v, w;
        asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(v), "=r"(w) : "r"(addr));
        d[0] = (T)(v & 0xffffu);
        d[1] = (T)(v >> 16);
        d[2] = (T)(w & 0xffffu);
        d[3] = (T)(w >> 16);
    }
};

// sum of one double per consumer thread, fixed order; result valid in consumer thread 0
__device__ __forceinline__ double consumer_block_sum(double v, double* scratch /* >= 8 doubles */, int ctid) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((ctid & 31) == 0) scratch[ctid >> 5] = v;
    consumer_bar();
    double s = 0.0;
    if (ctid == 0) {
#pragma unroll
        for (int w = 0; w < kConsumers / 32; ++w) s += scratch[w];
    }
    consumer_bar();
    return s;
}
__device__ __forceinline__ double consumer_block_max(double v, double* scratch, int ctid) {
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((ctid & 31) == 0) scratch[ctid >> 5] = v;
    consumer_bar();
    double s = 0.0;
    if (ctid == 0) {
#pragma unroll
        for (int w = 0; w < kConsumers / 32; ++w) s = fmax(s, scratch[w]);
    }
    consumer_bar();
    return s;
}

// Common CTA set-up: barriers and the tile share of this CTA.
struct CtaCtx {
    SmemCtl* ctl;
    int n_my;          // tiles this CTA owns (global tiles blockIdx.x, blockIdx.x + gridDim.x, ...)
    int last_rows;     // rows in the last global tile
    int warp, lane, ctid;
};

__device__ __forceinline__ void cta_setup(const Geom& g, unsigned char* smem, CtaCtx& c) {
    c.ctl = reinterpret_cast<SmemCtl*>(smem);
    c.warp = threadIdx.x >> 5;
    c.lane = threadIdx.x & 31;
    c.ctid = threadIdx.x;
    const int first = part_id(g);
    c.n_my = (g.n_tiles > first) ? (g.n_tiles - first + g.n_parts - 1) / g.n_parts : 0;
    c.last_rows = (int)(g.M - (long long)(g.n_tiles - 1) * g.tile_rows);
    if (threadIdx.x == 0) {
#pragma unroll
        for (int s = 0; s < kStages; ++s) {
            mbar_init(smem_u32(&c.ctl->full[s]), 1);
            mbar_init(smem_u32(&c.ctl->empty[s]), kConsumers / 32);
        }
        mbar_fence_init();
    }
}

// Rolling view of the stage ring (all 32-bit): tile counter, stage, barrier parity, stage address, global tile.
struct Ring {
    int it, s, gtile;
    unsigned parity;
    uint32_t sb;
    __device__ __forceinline__ void init(const Geom& g, uint32_t stages32) { it = 0; s = 0; parity = 0; sb = stages32; gtile = part_id(g); }
    __device__ __forceinline__ void advance(const Geom& g, uint32_t stages32) {
        ++it;
        gtile += g.n_parts;
        if (++s == n_stages(g)) { s = 0; parity ^= 1u; sb = stages32; }
        else sb += g.stage_bytes;
    }
    __device__ __forceinline__ int rows(const Geom& g, const CtaCtx& c) const { return gtile == g.n_tiles - 1 ? c.last_rows : g.tile_rows; }
};

// Producer duty is rotated over the warps (tile t is requested by warp t mod 8, between its own tiles), so no
// single warp lags behind.  Requests run (stages - 2) tiles ahead of consumption: the stage being
// refilled was released a full tile ago, so the requesting warp practically never waits on `empty`.
__device__ __forceinline__ void produce_next(const Geom& g, const FitDev& f, const CtaCtx& c, Ring& pr, uint32_t stages32, int nsrc) {
    if (pr.it < c.n_my && c.warp == (pr.it & (kConsumers / 32 - 1))) {
        mbar_wait(smem_u32(&c.ctl->empty[pr.s]), pr.parity ^ 1u);
        const int nrows = pr.rows(g, c);
        const uint32_t full = smem_u32(&c.ctl->full[pr.s]);
        if (nrows == g.tile_rows && f.rows == nullptr) {
            if (c.lane == 0) {
                const TileSrc* src = c.ctl->src;
                unsigned tx = 0;
#pragma unroll
                for (int k = 0; k < kMaxSrc; ++k)
                    if (k < nsrc && src[k].base != nullptr) tx += g.tile_tx[k];
                mbar_arrive_expect_tx(full, tx);
#pragma unroll
                for (int k = 0; k < kMaxSrc; ++k)
                    if (k < nsrc && src[k].base != nullptr)
                        bulk_g2s(pr.sb + src[k].off, src[k].base + (unsigned long long)pr.gtile * g.tile_tx[k], g.tile_tx[k], full);
            }
            __syncwarp();
        } else {
            produce_tile(c.ctl->src, nsrc, f.rows, (long long)pr.gtile * g.tile_rows, nrows,
                         reinterpret_cast<char*>(__cvta_shared_to_generic(pr.sb)), full, c.lane);
        }
    }
    pr.advance(g, stages32);
}

// Register row [R_trunc row (Kp entries, zero padded) | u row (ldu entries, zero padded)] is fetched as
// NCH two-element chunks; chunk i lives at  stage + off[i] + row * pitch[i].  Chunks beyond the real row
// alias chunk 0 (their alpha rows are zero, so they contribute nothing).
template <int NCH>
struct ChunkMap {
    unsigned off[NCH];
    unsigned pitch[NCH];
};
template <typename T, int NCH>
__device__ __forceinline__ void make_chunk_map(const Geom& g, ChunkMap<NCH>& m) {
    const int nR = g.Kp >> 1, nU = g.nup >> 1;
#pragma unroll
    for (int i = 0; i < NCH; ++i) {
        if (i < nR) { m.off[i] = g.offR + i * 2 * (unsigned)sizeof(T); m.pitch[i] = (unsigned)(g.ldr * sizeof(T)); }
        else if (i < nR + nU) { m.off[i] = g.offU + (i - nR) * 2 * (unsigned)sizeof(T); m.pitch[i] = (unsigned)(g.ldu * sizeof(T)); }
        else if (nR > 0) { m.off[i] = g.offR; m.pitch[i] = (unsigned)(g.ldr * sizeof(T)); }
        else { m.off[i] = g.offU; m.pitch[i] = (unsigned)(g.ldu * sizeof(T)); }
    }
}
// alpha row that register-row entry i multiplies (-1: padding)
__device__ __forceinline__ int alpha_row_of(const Geom& g, int i) {
    if (i < g.Kp) return i < g.K ? i : -1;
    const int q = i - g.Kp;
    return q < g.nu ? g.K + q : -1;
}

// ------------------------------------------------------------------------------------------------
// Minimum CTAs per SM of the streaming passes (__launch_bounds__); make_plan sizes their ring for the same occupancy.
__host__ __device__ constexpr int pass_min_blocks(int ktb) { return ktb <= 8 ? 2 : 1; }      // cost_kernel, alpha_pass_kernel
__host__ __device__ constexpr int u_pass_min_blocks(int kb, int nub, int c) { return (kb + 2 * nub) * c <= 24 ? 2 : 1; }

// cost / set-up pass
template <typename T, typename WT, int KTB, int C, bool INITIAL>
__global__ void __launch_bounds__(kThreads, pass_min_blocks(KTB)) cost_kernel(const PassArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NCH = KTB / 2;
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    CtaCtx c;
    cta_setup(g, smem, c);
    unsigned char* stages = smem + kCtlBytes;
    const uint32_t stages32 = smem_u32(stages);
    const int ucur = st->u_cur, acur = st->a_cur;
    const T* Acur = reinterpret_cast<const T*>(f.A) + (size_t)acur * g.Kt * g.N;
    const char* Ucur = f.U + (size_t)ucur * g.uslot_bytes;

    double cost = 0.0, ssq_r = 0.0, ssq_u = 0.0, dmx = 0.0;
    constexpr int NSRC = 4;
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(T), g.offX, 1, (unsigned char)(g.row_bulk & 1u), 0};
        src[1] = {f.D, g.ldd * (long long)sizeof(WT), g.offD, 1, (unsigned char)((g.row_bulk >> 1) & 1u), 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(T), g.offR, 1, (unsigned char)((g.row_bulk >> 2) & 1u), 0};
        src[3] = {Ucur, g.ldu * (long long)sizeof(T), g.offU, 0, 0, 0};
    }
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, NSRC);
    {
        const int tc = c.ctid % g.ntc, gr = c.ctid / g.ntc;
        const bool colvalid = C * tc < g.N;
        const int j0 = colvalid ? C * tc : 0;
        T at[KTB][C];
#pragma unroll
        for (int k = 0; k < KTB; ++k) {
            const int ar = alpha_row_of(g, k);
#pragma unroll
            for (int cc = 0; cc < C; ++cc) at[k][cc] = (ar >= 0 && j0 + cc < g.N) ? Acur[(size_t)ar * g.N + j0 + cc] : (T)0;
        }
        ChunkMap<NCH> cm;
        make_chunk_map<T, NCH>(g, cm);
        const unsigned xoff = g.offX + (unsigned)(j0 * sizeof(T)), xpitch = (unsigned)(g.ldx * sizeof(T));
        const unsigned doff = g.offD + (unsigned)(j0 * sizeof(WT)), dpitch = (unsigned)(g.ldd * sizeof(WT));
        for (; cr.it < c.n_my; cr.advance(g, stages32)) {
            produce_next(g, f, c, pr, stages32, NSRC);
            mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
            const uint32_t sb = cr.sb;
            const int nrows = cr.rows(g, c);
            if (colvalid) {
                for (int r = gr; r < nrows; r += g.rg) {
                    T rrow[KTB];
#pragma unroll
                    for (int i = 0; i < NCH; ++i) lds2(sb + cm.off[i] + r * cm.pitch[i], rrow[2 * i], rrow[2 * i + 1]);
                    if (INITIAL && tc == 0) {
#pragma unroll
                        for (int k = 0; k < KTB; ++k) {
                            const double v = (double)rrow[k];
                            const int ar = alpha_row_of(g, k);
                            if (ar >= 0 && ar < g.K) ssq_r = fma(v, v, ssq_r);
                            else if (ar >= g.K) ssq_u = fma(v, v, ssq_u);
                        }
                    }
                    T x[C], d[C], p[C];
                    ldsC<T, C>(sb + xoff + r * xpitch, x);
                    WLoad<T, WT, C>::ld(sb + doff + r * dpitch, d);
                    // two independent chains per column (even / odd entries) halve the dependent-FMA latency
                    T pe[C], po[C];
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) { pe[cc] = rrow[0] * at[0][cc]; po[cc] = rrow[1] * at[1][cc]; }
#pragma unroll
                    for (int k = 2; k < KTB; k += 2)
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) {
                            pe[cc] = fma_t<T>(rrow[k], at[k][cc], pe[cc]);
                            po[cc] = fma_t<T>(rrow[k + 1], at[k + 1][cc], po[cc]);
                        }
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) p[cc] = pe[cc] + po[cc];
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) {
                        const double e = (double)(x[cc] - p[cc]);
                        cost = fma((double)d[cc] * e, e, cost);
                        if (INITIAL) dmx = fmax(dmx, (double)d[cc]);
                    }
                }
            }
            __syncwarp();
            if (c.lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));
        }
    }
    __syncthreads();
    // CTA partial record: [cost, ssq_rk, ssq_u, dmax]
    double* scratch = reinterpret_cast<double*>(stages);
    double* rec = scratch + 16;
    if (c.warp < kConsumers / 32) {
        const double s0 = consumer_block_sum(cost, scratch, c.ctid);
        double s1 = 0.0, s2 = 0.0, s3 = 0.0;
        if (INITIAL) {
            s1 = consumer_block_sum(ssq_r, scratch, c.ctid);
            s2 = consumer_block_sum(ssq_u, scratch, c.ctid);
            s3 = consumer_block_max(dmx, scratch, c.ctid);
        }
        if (c.ctid == 0) {
            double* p = f.part + (size_t)part_id(g) * g.part_stride;
            p[0] = s0; p[1] = s1; p[2] = s2; p[3] = s3;
        }
    }
    // dmax needs a max, not a sum: it travels through slot 3 of every record and is re-derived below.
    if (!hier_reduce(g, f, rec, 3, &c.ctl->flag)) return;
    if (threadIdx.x == 0) {
        const double cf = rec[0];
        if (INITIAL) {
            double dm = 0.0;
            for (int p = 0; p < g.n_parts; ++p) dm = fmax(dm, __ldcg(&f.part[(size_t)p * g.part_stride + 3]));
            st->dmax = dm;
            st->dmax2 = dm * dm;
            st->ssq_rk = rec[1];
            st->ssq_u = rec[2];
            // ||alpha[-n_u:]||_F^2 (deconvolution.py:198): tiny, done serially in row-major order
            double sa = 0.0;
            for (int q = 0; q < g.nu; ++q)
                for (int j = 0; j < g.N; ++j) {
                    const double v = (double)Acur[(size_t)(g.K + q) * g.N + j];
                    sa = fma(v, v, sa);
                }
            const double na = sqrt(sa), nr = sqrt(rec[1] + rec[2]);
            st->l_w = (na * na) * st->dmax2;
            st->l_w_old = st->l_w;
            st->l_h = (nr * nr) * st->dmax2;
            st->l_h_old = st->l_h;
            st->a1 = 1.0;
            st->a2 = 1.0;
            st->cf = cf;
            st->cf_prev = cf;
            st->n_outer = 0;
            st->t_u = 0;
            st->t_a = 0;
            if (f.trace && f.trace_cap > 0) f.trace[0] = cf;
        } else {
            const double prev = st->cf;
            st->cf_prev = prev;
            st->cf = cf;
            const int n = st->n_outer + 1;
            st->n_outer = n;
            if (f.trace && n < f.trace_cap) f.trace[n] = cf;
            if (fabs(cf - prev) < a.tol) st->done = 1;      // deconvolution.py:220
            if (!(cf == cf)) st->done = 3;                    // NaN guard
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Segmented reduction of NV doubles per lane over aligned groups of L lanes (L power of two <= 32).
// Transposed butterfly: while more than one value is left, each step halves the number of values a lane
// carries (small offsets first), then plain xor-adds cover the remaining offsets.  Deterministic.
// On return lane l holds the group totals of slots  slot_base + i,  i < count.
template <int NV>
__device__ __forceinline__ void seg_reduce(double (&v)[NV], int L, int lane, int& slot_base, int& count) {
    int n = NV;
    slot_base = 0;
#pragma unroll
    for (int s = 0; s < 5; ++s) {
        const int o = 1 << s;
        if (o < L) {
            const int half = NV >> (s + 1);          // compile-time: values kept when every earlier step ran
            if (half >= 1) {
                const bool up = (lane & o) != 0;
#pragma unroll
                for (int i = 0; i < (NV >> (s + 1)); ++i) {
                    const double send = up ? v[i] : v[i + half];
                    const double keep = up ? v[i + half] : v[i];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
                }
                n = half;
                slot_base += up ? half : 0;
            } else {
                v[0] += __shfl_xor_sync(0xffffffffu, v[0], o);
            }
        }
    }
    count = n;
}

// U pass: u <- clip(u_t + ((d o (x - Rk a_k - u_g a_u)) a_u^T) / l_w, 0, 1),  u_t = u + beta (u - u_prev)
// (u_g = u_t in update_u:88, u_g = u in unsupervised_deconv:163)
template <typename T, typename WT, int KB, int NUB, int C, int RPT>
__global__ void __launch_bounds__(kThreads, u_pass_min_blocks(KB, NUB, C)) u_pass_kernel(const PassArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NV = RPT * NUB;
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    CtaCtx c;
    cta_setup(g, smem, c);
    unsigned char* stages = smem + kCtlBytes;
    const uint32_t stages32 = smem_u32(stages);
    const int ucur = st->u_cur, acur = st->a_cur;
    const double a_prev = st->a1, l_w = st->l_w, l_w_old = st->l_w_old;
    const double a_next = next_momentum(a_prev);
    const T beta = (T)extrap_beta(a_prev, a_next, l_w_old, l_w);
    const T lw = (T)l_w;
    const T* Acur = reinterpret_cast<const T*>(f.A) + (size_t)acur * g.Kt * g.N;
    const char* Ucur = f.U + (size_t)ucur * g.uslot_bytes;
    char* Uprev = f.U + (size_t)(ucur ^ 1) * g.uslot_bytes;      // read as u_prev, overwritten with the new u
    const bool at_current = (g.mode == 2);

    double ssq_u = 0.0;
    constexpr int NSRC = 5;
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(T), g.offX, 1, (unsigned char)(g.row_bulk & 1u), 0};
        src[1] = {f.D, g.ldd * (long long)sizeof(WT), g.offD, 1, (unsigned char)((g.row_bulk >> 1) & 1u), 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(T), g.offR, 1, (unsigned char)((g.row_bulk >> 2) & 1u), 0};
        src[3] = {Ucur, g.ldu * (long long)sizeof(T), g.offU, 0, 0, 0};
        src[4] = {Uprev, g.ldu * (long long)sizeof(T), g.offUp, 0, 0, 0};
    }
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, NSRC);
    {
        const int tc = c.ctid % g.ntc, gr = c.ctid / g.ntc;
        const bool colvalid = C * tc < g.N;
        const int j0 = colvalid ? C * tc : 0;
        const int L = min(g.ntc, 32);
        const int wpr = (g.ntc + 31) / 32;           // warps per row
        const int wir = tc >> 5;                      // my warp's index within the row
        T ak[KB][C];     // known block of alpha, my columns
        T au[NUB][C];    // unknown block (zero for padding columns: they add nothing to the row sums)
#pragma unroll
        for (int k = 0; k < KB; ++k)
#pragma unroll
            for (int cc = 0; cc < C; ++cc) ak[k][cc] = (k < g.K && colvalid && j0 + cc < g.N) ? Acur[(size_t)k * g.N + j0 + cc] : (T)0;
#pragma unroll
        for (int q = 0; q < NUB; ++q)
#pragma unroll
            for (int cc = 0; cc < C; ++cc) au[q][cc] = (q < g.nu && colvalid && j0 + cc < g.N) ? Acur[(size_t)(g.K + q) * g.N + j0 + cc] : (T)0;
        const unsigned xoff = g.offX + (unsigned)(j0 * sizeof(T)), xpitch = (unsigned)(g.ldx * sizeof(T));
        const unsigned doff = g.offD + (unsigned)(j0 * sizeof(WT)), dpitch = (unsigned)(g.ldd * sizeof(WT));
        const unsigned rpitch = (unsigned)(g.ldr * sizeof(T)), upitch = (unsigned)(g.ldu * sizeof(T));
        const int nRch = g.Kp >> 1, nUch = g.nup >> 1;
        // cross-warp combine buffer (rows spanning several warps): [2][tile_rows][nu][wpr]
        double* red = reinterpret_cast<double*>(stages + (size_t)kStages * g.stage_bytes);

        for (; cr.it < c.n_my; cr.advance(g, stages32)) {
            produce_next(g, f, c, pr, stages32, NSRC);
            mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
            const uint32_t sb = cr.sb;
            const int nrows = cr.rows(g, c);
            double* redt = red + (size_t)(cr.it & 1) * g.tile_rows * g.nu * wpr;
            T* Uout = reinterpret_cast<T*>(Uprev) + (size_t)cr.gtile * g.tile_rows * g.ldu;

            double gp[NV];
            T utk[RPT][NUB];
#pragma unroll
            for (int rb = 0; rb < RPT; ++rb) {
                const int r = gr + rb * g.rg;
                const bool live = (rb < g.rpt) && (r < nrows);
                const int rr = live ? r : 0;                      // dead rows recompute row 0; their slots are never stored
                T rk[KB], ug[NUB];
#pragma unroll
                for (int i = 0; i < KB / 2; ++i) {
                    const int ii = i < nRch ? i : 0;
                    lds2(sb + g.offR + ii * 2 * (unsigned)sizeof(T) + rr * rpitch, rk[2 * i], rk[2 * i + 1]);
                }
#pragma unroll
                for (int i = 0; i < NUB / 2; ++i) {
                    const int ii = i < nUch ? i : 0;
                    T u0, u1, p0, p1;
                    lds2(sb + g.offU + ii * 2 * (unsigned)sizeof(T) + rr * upitch, u0, u1);
                    lds2(sb + g.offUp + ii * 2 * (unsigned)sizeof(T) + rr * upitch, p0, p1);
                    utk[rb][2 * i] = u0 + beta * (u0 - p0);
                    utk[rb][2 * i + 1] = u1 + beta * (u1 - p1);
                    ug[2 * i] = at_current ? u0 : utk[rb][2 * i];
                    ug[2 * i + 1] = at_current ? u1 : utk[rb][2 * i + 1];
                }
                T x[C], d[C], pk[C], pu[C];
                ldsC<T, C>(sb + xoff + rr * xpitch, x);
                WLoad<T, WT, C>::ld(sb + doff + rr * dpitch, d);
                T pk1[C];
#pragma unroll
                for (int cc = 0; cc < C; ++cc) { pk[cc] = rk[0] * ak[0][cc]; pk1[cc] = rk[1] * ak[1][cc]; pu[cc] = (T)0; }
#pragma unroll
                for (int k = 2; k < KB; k += 2)
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) {
                        pk[cc] = fma_t<T>(rk[k], ak[k][cc], pk[cc]);
                        pk1[cc] = fma_t<T>(rk[k + 1], ak[k + 1][cc], pk1[cc]);
                    }
#pragma unroll
                for (int cc = 0; cc < C; ++cc) pk[cc] = pk[cc] + pk1[cc];
#pragma unroll
                for (int q = 0; q < NUB; ++q)
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) pu[cc] = fma_t<T>(ug[q], au[q][cc], pu[cc]);
                T w[C];
#pragma unroll
                for (int cc = 0; cc < C; ++cc) w[cc] = d[cc] * ((x[cc] - pk[cc]) - pu[cc]);   // (X - R_trunc a_k) - u a_u, :88
#pragma unroll
                for (int q = 0; q < NUB; ++q) {
                    T acc = w[0] * au[q][0];
#pragma unroll
                    for (int cc = 1; cc < C; ++cc) acc = fma_t<T>(w[cc], au[q][cc], acc);
                    gp[rb * NUB + q] = (double)acc;
                }
            }
            // row sums over the column threads
            int slot_base, count;
            seg_reduce<NV>(gp, L, c.lane, slot_base, count);
            const bool owner = ((c.lane & (L - 1)) & ~(NV - 1)) == 0;     // lanes sharing a slot set: one writes
            if (wpr == 1) {
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    if (i < count) {
                        const int slot = slot_base + i;
                        const int rb = slot / NUB, q = slot - rb * NUB;
                        const int r = gr + rb * g.rg;
                        if (owner && rb < g.rpt && r < nrows && q < g.nu) {
                            T utq = (T)0;
#pragma unroll
                            for (int b2 = 0; b2 < RPT; ++b2)
#pragma unroll
                                for (int q2 = 0; q2 < NUB; ++q2)
                                    if (b2 == rb && q2 == q) utq = utk[b2][q2];
                            T un = utq + (T)gp[i] / lw;
                            un = un < (T)0 ? (T)0 : (un > (T)1 ? (T)1 : un);
                            Uout[(size_t)r * g.ldu + q] = un;
                            ssq_u = fma((double)un, (double)un, ssq_u);
                        }
                    }
                }
            } else {
#pragma unroll
                for (int i = 0; i < NV; ++i) {
                    if (i < count) {
                        const int slot = slot_base + i;
                        const int rb = slot / NUB, q = slot - rb * NUB;
                        const int r = gr + rb * g.rg;
                        if (owner && rb < g.rpt && r < nrows && q < g.nu) redt[((size_t)r * g.nu + q) * wpr + wir] = gp[i];
                    }
                }
                // only the warps of this row group meet: named barrier 1 + gr, ntc threads
                asm volatile("bar.sync %0, %1;" ::"r"(1 + gr), "r"(g.ntc) : "memory");
                const T* sU = reinterpret_cast<const T*>(stages + (size_t)cr.s * g.stage_bytes + g.offU);
                const T* sUp = reinterpret_cast<const T*>(stages + (size_t)cr.s * g.stage_bytes + g.offUp);
                for (int e2 = tc; e2 < g.rpt * g.nu; e2 += g.ntc) {
                    const int rb = e2 / g.nu, q = e2 - rb * g.nu;
                    const int r = gr + rb * g.rg;
                    if (r >= nrows) continue;
                    const int e = r * g.nu + q;
                    double v = 0.0;
                    for (int w2 = 0; w2 < wpr; ++w2) v += redt[(size_t)e * wpr + w2];
                    const T u = sU[(size_t)r * g.ldu + q], up = sUp[(size_t)r * g.ldu + q];
                    const T utq = u + beta * (u - up);
                    T un = utq + (T)v / lw;
                    un = un < (T)0 ? (T)0 : (un > (T)1 ? (T)1 : un);
                    Uout[(size_t)r * g.ldu + q] = un;
                    ssq_u = fma((double)un, (double)un, ssq_u);
                }
            }
            __syncwarp();
            if (c.lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));
        }
    }
    __syncthreads();
    double* scratch = reinterpret_cast<double*>(stages);
    double* rec = scratch + 16;
    if (c.warp < kConsumers / 32) {
        const double s0 = consumer_block_sum(ssq_u, scratch, c.ctid);
        if (c.ctid == 0) f.part[(size_t)part_id(g) * g.part_stride] = s0;
    }
    if (!hier_reduce(g, f, rec, 1, &c.ctl->flag)) return;
    if (threadIdx.x == 0) {
        st->a1 = a_next;
        st->t_u += 1;
        st->l_w_old = l_w;                                   // deconvolution.py:89
        st->u_cur = ucur ^ 1;
        st->ssq_u = rec[0];
        const double nr = sqrt(st->ssq_rk + rec[0]);
        st->l_h = (nr * nr) * st->dmax2;                     // deconvolution.py:212 (read by the alpha steps only)
    }
}

// ------------------------------------------------------------------------------------------------
// simplex projection of one column held in v[0..p) (deconvolution.py:21-37); returns false on NaN
__device__ __forceinline__ bool project_simplex(double* v, int p) {
    double u[kMaxKt];
    for (int i = 0; i < p; ++i) u[i] = v[i];
    for (int i = 1; i < p; ++i) {          // insertion sort, descending
        const double key = u[i];
        int j = i - 1;
        while (j >= 0 && u[j] < key) { u[j + 1] = u[j]; --j; }
        u[j + 1] = key;
    }
    double cs = 0.0, theta = 0.0;
    int rho = -1;
    for (int j = 0; j < p; ++j) {
        cs += u[j];
        const double pi = cs - 1.0;
        if (u[j] - pi / (double)(j + 1) > 0.0) { rho = j; theta = pi / (double)(j + 1); }
    }
    if (rho < 0) return false;
    for (int i = 0; i < p; ++i) v[i] = fmax(v[i] - theta, 0.0);
    return true;
}

// alpha pass: G = R^T (d o (x - R a_eval)); last CTA applies the projected-gradient or Frank-Wolfe step
template <typename T, typename WT, int KTB, int C>
__global__ void __launch_bounds__(kThreads, pass_min_blocks(KTB)) alpha_pass_kernel(const PassArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NCH = KTB / 2;
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    CtaCtx c;
    cta_setup(g, smem, c);
    unsigned char* stages = smem + kCtlBytes;
    const uint32_t stages32 = smem_u32(stages);
    const bool fw = (a.flags & kFlagFW) != 0;
    const int ucur = st->u_cur, acur = st->a_cur;
    const double a_prev = st->a2, l_h = st->l_h, l_h_old = st->l_h_old;
    const double a_next = next_momentum(a_prev);
    const double beta_d = fw ? 0.0 : extrap_beta(a_prev, a_next, l_h_old, l_h);
    const T beta = (T)beta_d;
    T* Acur = reinterpret_cast<T*>(f.A) + (size_t)acur * g.Kt * g.N;
    T* Aprev = reinterpret_cast<T*>(f.A) + (size_t)(acur ^ 1) * g.Kt * g.N;
    const char* Ucur = f.U + (size_t)ucur * g.uslot_bytes;

    const int tc = c.ctid % g.ntc, gr = c.ctid / g.ntc;
    const bool colvalid = (c.ctid < kConsumers) && (C * tc < g.N);
    const int j0 = colvalid ? C * tc : 0;
    T G[KTB][C];
#pragma unroll
    for (int k = 0; k < KTB; ++k)
#pragma unroll
        for (int cc = 0; cc < C; ++cc) G[k][cc] = (T)0;

    constexpr int NSRC = 4;
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(T), g.offX, 1, (unsigned char)(g.row_bulk & 1u), 0};
        src[1] = {f.D, g.ldd * (long long)sizeof(WT), g.offD, 1, (unsigned char)((g.row_bulk >> 1) & 1u), 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(T), g.offR, 1, (unsigned char)((g.row_bulk >> 2) & 1u), 0};
        src[3] = {Ucur, g.ldu * (long long)sizeof(T), g.offU, 0, 0, 0};
    }
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, NSRC);
    {
        T at[KTB][C];    // evaluation point: alpha_temp (PG) or alpha (FW)
#pragma unroll
        for (int k = 0; k < KTB; ++k) {
            const int ar = alpha_row_of(g, k);
#pragma unroll
            for (int cc = 0; cc < C; ++cc) {
                T v = (T)0;
                if (ar >= 0 && colvalid && j0 + cc < g.N) {
                    const T ac = Acur[(size_t)ar * g.N + j0 + cc];
                    v = ac;
                    if (!fw) v = ac + beta * (ac - Aprev[(size_t)ar * g.N + j0 + cc]);
                }
                at[k][cc] = v;
            }
        }
        ChunkMap<NCH> cm;
        make_chunk_map<T, NCH>(g, cm);
        const unsigned xoff = g.offX + (unsigned)(j0 * sizeof(T)), xpitch = (unsigned)(g.ldx * sizeof(T));
        const unsigned doff = g.offD + (unsigned)(j0 * sizeof(WT)), dpitch = (unsigned)(g.ldd * sizeof(WT));
        for (; cr.it < c.n_my; cr.advance(g, stages32)) {
            produce_next(g, f, c, pr, stages32, NSRC);
            mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
            const uint32_t sb = cr.sb;
            const int nrows = cr.rows(g, c);
            if (colvalid) {
                for (int r = gr; r < nrows; r += g.rg) {
                    T rrow[KTB];
#pragma unroll
                    for (int i = 0; i < NCH; ++i) lds2(sb + cm.off[i] + r * cm.pitch[i], rrow[2 * i], rrow[2 * i + 1]);
                    T x[C], d[C], p[C];
                    ldsC<T, C>(sb + xoff + r * xpitch, x);
                    WLoad<T, WT, C>::ld(sb + doff + r * dpitch, d);
                    // two independent chains per column (even / odd entries) halve the dependent-FMA latency
                    T pe[C], po[C];
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) { pe[cc] = rrow[0] * at[0][cc]; po[cc] = rrow[1] * at[1][cc]; }
#pragma unroll
                    for (int k = 2; k < KTB; k += 2)
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) {
                            pe[cc] = fma_t<T>(rrow[k], at[k][cc], pe[cc]);
                            po[cc] = fma_t<T>(rrow[k + 1], at[k + 1][cc], po[cc]);
                        }
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) p[cc] = pe[cc] + po[cc];
                    T w[C];
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) w[cc] = d[cc] * (x[cc] - p[cc]);
#pragma unroll
                    for (int k = 0; k < KTB; ++k)
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) G[k][cc] = fma_t<T>(rrow[k], w[cc], G[k][cc]);
                }
            }
            __syncwarp();
            if (c.lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));
        }
    }
    __syncthreads();
    // combine the row groups of this CTA in fixed order, then publish the CTA partial [Kt][N]
    double* scratch = reinterpret_cast<double*>(stages);
    const int KN = g.Kt * g.N;
    if (c.warp < kConsumers / 32) {
        for (int gg = 0; gg < g.rg; ++gg) {
            if (gr == gg && colvalid) {
#pragma unroll
                for (int k = 0; k < KTB; ++k) {
                    const int ar = alpha_row_of(g, k);
#pragma unroll
                    for (int cc = 0; cc < C; ++cc)
                        if (ar >= 0 && j0 + cc < g.N) {
                            double* p = &scratch[(size_t)ar * g.N + j0 + cc];
                            *p = (gg == 0) ? (double)G[k][cc] : (*p + (double)G[k][cc]);
                        }
                }
            }
            consumer_bar();
        }
        double* part = f.part + (size_t)part_id(g) * g.part_stride;
        for (int e = c.ctid; e < KN; e += kConsumers) part[e] = scratch[e];
    }
    if (!hier_reduce(g, f, scratch, KN, &c.ctl->flag)) return;

    // ---- last CTA: apply the step on the Kt x N gradient held in scratch
    double* colred = scratch + KN;        // per-column ||alpha_unk||^2 contributions
    int bad = 0;
    for (int j = threadIdx.x; j < g.N; j += blockDim.x) {
        double v[kMaxKt];
        double sa = 0.0;
        if (!fw) {
            for (int k = 0; k < g.Kt; ++k) {
                const T ac = Acur[(size_t)k * g.N + j], ap = Aprev[(size_t)k * g.N + j];
                const T atv = ac + beta * (ac - ap);
                v[k] = (double)(atv + (T)(scratch[(size_t)k * g.N + j]) / (T)l_h);
            }
            if (!project_simplex(v, g.Kt)) bad = 1;
            else
                for (int k = 0; k < g.Kt; ++k) Aprev[(size_t)k * g.N + j] = (T)v[k];   // becomes the current slot
            for (int q = 0; q < g.nu; ++q) sa = fma(v[g.K + q], v[g.K + q], sa);
        } else {
            // gradient = -G; vertex = FIRST argmin of each block (np.argmin), deconvolution.py:286-299
            const double pj = f.purity[j];
            const double gamma = 2.0 / (double)(a.k_inner + 2);
            int i1 = 0, i2 = 0;
            double m1 = 0.0, m2 = 0.0;
            for (int k = 0; k < g.K; ++k) {
                const double gk = -scratch[(size_t)k * g.N + j];
                if (k == 0 || gk < m1) { m1 = gk; i1 = k; }
            }
            for (int q = 0; q < g.nu; ++q) {
                const double gq = -scratch[(size_t)(g.K + q) * g.N + j];
                if (q == 0 || gq < m2) { m2 = gq; i2 = q; }
            }
            for (int k = 0; k < g.Kt; ++k) {
                const double s = (k < g.K) ? ((k == i1) ? pj : 0.0) : ((k - g.K == i2) ? (1.0 - pj) : 0.0);
                const double an = (1.0 - gamma) * (double)Acur[(size_t)k * g.N + j] + gamma * s;
                Acur[(size_t)k * g.N + j] = (T)an;
                if (k >= g.K) sa = fma(an, an, sa);
            }
        }
        colred[j] = sa;
    }
    if (bad) st->done = 3;
    __syncthreads();
    if (threadIdx.x == 0) {
        double sa = 0.0;
        for (int j = 0; j < g.N; ++j) sa += colred[j];
        const double na = sqrt(sa);
        st->l_w = (na * na) * st->dmax2;                 // deconvolution.py:216 / :327 (read by the U steps only)
        if (!fw) {
            st->a2 = a_next;
            st->t_a += 1;
            st->l_h_old = l_h;                           // deconvolution.py:101
            st->a_cur = acur ^ 1;
        }
    }
}

}  // namespace dmf
