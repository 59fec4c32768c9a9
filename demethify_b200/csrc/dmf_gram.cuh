// dmf_gram.cuh — "Gram-form" engine: the same outer iteration as deconvolution.py:206-221 / :320-335, restated so that
// the n_iter2 inner iterations of update_u (:82-89) and update_alpha (:94-101) / frank_wolfe_nmf (:285-299) run on
// small sufficient statistics instead of re-streaming X and d_x 2 * n_iter2 times (SURVEY.md 7.1 #1-#4):
//
//   U step   (alpha frozen)  gradient row m:  (d o (c - u_g a_u)) a_u^T  =  b_m - H_m u_g        c = x - R_trunc a_k
//                            b_m[q]    = sum_j d_mj c_mj a_u[q,j]          (n_u values per row)
//                            H_m[q,q'] = sum_j d_mj a_u[q,j] a_u[q',j]     (n_u (n_u+1)/2 values per row)
//   alpha step (R frozen)    gradient col j:  R^T (d o (x - R a_t))      =  bx_j - G_j a_t
//                            G_j = R^T diag(d_.j) R  (Kt x Kt),  bx_j = R^T (d_.j o x_.j)
//
//   rowgram_kernel     ONE streaming pass: b_m, H_m for every row + cost_f_w of the current iterate (direct form,
//                      so the |cf - cf_0| < tol test sees the same number as the reference-shaped cost pass)
//   u_inner_kernel     n_iter2 update_u iterations per row on (b_m, H_m): row-local, no streaming of X
//   gram_panel_kernel  ONE streaming pass: the blocks of G_j, bx_j that involve u (the known x known block and
//                      the known part of bx are invariant and computed once at set-up)
//   alpha_inner_kernel n_iter2 update_alpha (with simplex projection) or Frank-Wolfe iterations per sample on (G_j, bx_j)
// plus, for bootstrap resamples in multiplicity form (shared source matrices, per-position u through a CSR):
//   u_inner_mult_kernel / usum_kernel / cost_cross_kernel and the MULT variant of gram_panel_kernel,
// and, for CpG rows sharded over GPUs: finalize_cost_kernel (set-up / termination on all-reduced sums) and
//   peer_allreduce_kernel (the all-reduce itself, over NVLink peer memory).
//
// An outer iteration is 2 streaming passes + 2 small kernels instead of 2 n_iter2 + 1 streaming passes.  The sums are
// re-associated with respect to the reference (fp64, fixed order), which moves alpha by ~1e-15; the termination test
// uses the directly computed cost.  Parity is pinned by the same golden vectors as the reference-shaped passes.
#pragma once
#include "dmf_kernels.cuh"

namespace dmf {

// np.clip(., 0, 1) of deconvolution.py:88 as two min/max instructions (a NaN would become 0 here; non-finite inputs are
// caught by the simplex projection of the alpha step, which sees the same poisoned statistics)
__device__ __forceinline__ double clip01(double v) { return fmin(fmax(v, 0.0), 1.0); }
__device__ __forceinline__ float clip01(float v) { return fminf(fmaxf(v, 0.0f), 1.0f); }

__host__ __device__ constexpr int ng_of(int nub) { return nub + nub * (nub + 1) / 2; }
__host__ __device__ constexpr int pow2ceil(int v) { int p = 1; while (p < v) p <<= 1; return p; }
__host__ __device__ constexpr int tri_index(int q, int q2, int nub) { return q * nub - q * (q - 1) / 2 + (q2 - q); }   // q <= q2
// Minimum CTAs per SM of the rowgram and panel passes (__launch_bounds__); make_plan sizes their ring for the same occupancy.
// C == 4 is rowgram4_kernel (one CTA per SM).
__host__ __device__ constexpr int rowgram_min_blocks(int kb, int nub, int c, int rpt) {
    return c != 4 && (kb + 2 * nub) * c + 2 * pow2ceil(rpt * ng_of(nub)) <= 56 ? 2 : 1;
}
__host__ __device__ constexpr int panel_min_blocks(int pa, int pb, int c) { return pa * (pb + 1) * c <= 40 ? 2 : 1; }

// ------------------------------------------------------------------------------------------------
// rowgram pass.  Thread (row group gr, column thread tc) owns C adjacent columns and RPT rows of the tile; the per-row
// values [b (NUB) | H upper triangle] are summed over the column threads of a warp with the transposed butterfly and
// written per warp:  rowgram[row][warp-in-row][NG]  (u_inner_kernel adds the <= 8 per-warp partials in fixed order).
template <typename T, typename WT, int KB, int NUB, int C, int RPT, bool INITIAL>
__global__ void __launch_bounds__(kThreads, rowgram_min_blocks(KB, NUB, C, RPT)) rowgram_kernel(const PassArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NG = ng_of(NUB);
    constexpr int NVP = pow2ceil(RPT * NG);
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
        const int L = min(g.ntc, 32);
        const int wpr = (g.ntc + 31) / 32;
        const int wir = tc >> 5;
        T ak[KB > 0 ? KB : 1][C];
        T au[NUB][C];
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
        double* RG = f.rowgram;

        for (; cr.it < c.n_my; cr.advance(g, stages32)) {
            produce_next(g, f, c, pr, stages32, NSRC);
            mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
            const uint32_t sb = cr.sb;
            const int nrows = cr.rows(g, c);
            const long long grow0 = (long long)cr.gtile * g.tile_rows;

            double gp[NVP];
#pragma unroll
            for (int i = 0; i < NVP; ++i) gp[i] = 0.0;
#pragma unroll
            for (int rb = 0; rb < RPT; ++rb) {
                const int r = gr + rb * g.rg;
                const bool live = (rb < g.rpt) && (r < nrows);
                const int rr = live ? r : 0;                      // dead rows recompute row 0; never stored, never counted
                T rk[KB > 0 ? KB : 1], uc[NUB > 1 ? NUB : 2];
#pragma unroll
                for (int i = 0; i < KB / 2; ++i) {
                    const int ii = i < nRch ? i : 0;
                    lds2(sb + g.offR + ii * 2 * (unsigned)sizeof(T) + rr * rpitch, rk[2 * i], rk[2 * i + 1]);
                }
#pragma unroll
                for (int i = 0; i < (NUB + 1) / 2; ++i) {
                    const int ii = i < nUch ? i : 0;
                    lds2(sb + g.offU + ii * 2 * (unsigned)sizeof(T) + rr * upitch, uc[2 * i], uc[2 * i + 1]);
                }
                if (INITIAL && tc == 0 && live) {
#pragma unroll
                    for (int k = 0; k < KB; ++k)
                        if (k < g.K) ssq_r = fma((double)rk[k], (double)rk[k], ssq_r);
#pragma unroll
                    for (int q = 0; q < NUB; ++q)
                        if (q < g.nu) ssq_u = fma((double)uc[q], (double)uc[q], ssq_u);
                }
                T x[C], d[C], cres[C];
                ldsC<T, C>(sb + xoff + rr * xpitch, x);
                WLoad<T, WT, C>::ld(sb + doff + rr * dpitch, d);
                if (KB > 0) {
                    T pk[C], pk1[C];
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) { pk[cc] = rk[0] * ak[0][cc]; pk1[cc] = rk[KB > 1 ? 1 : 0] * ak[KB > 1 ? 1 : 0][cc]; }
#pragma unroll
                    for (int k = 2; k < KB; k += 2)
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) {
                            pk[cc] = fma_t<T>(rk[k], ak[k][cc], pk[cc]);
                            pk1[cc] = fma_t<T>(rk[k + 1], ak[k + 1][cc], pk1[cc]);
                        }
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) cres[cc] = x[cc] - (pk[cc] + pk1[cc]);     // c = x - R_trunc a_k
                } else {
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) cres[cc] = x[cc];
                }
                // cost of the current iterate: d * ((x - R_trunc a_k) - u a_u)^2
                if (live && colvalid) {
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) {
                        T pu = (T)0;
#pragma unroll
                        for (int q = 0; q < NUB; ++q) pu = fma_t<T>(uc[q], au[q][cc], pu);
                        const double e = (double)(cres[cc] - pu);
                        cost = fma((double)d[cc] * e, e, cost);
                        if (INITIAL) dmx = fmax(dmx, (double)d[cc]);
                    }
                }
                // b[q] and H[q][q'] partial sums over my columns (padding columns have au = 0)
#pragma unroll
                for (int q = 0; q < NUB; ++q) {
                    double bq = 0.0;
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) bq = fma((double)(d[cc] * cres[cc]), (double)au[q][cc], bq);
                    gp[rb * NG + q] = bq;
#pragma unroll
                    for (int q2 = q; q2 < NUB; ++q2) {
                        double h = 0.0;
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) h = fma((double)(d[cc] * au[q][cc]), (double)au[q2][cc], h);
                        gp[rb * NG + NUB + tri_index(q, q2, NUB) - 0] = h;
                    }
                }
            }
            int slot_base, count;
            seg_reduce<NVP>(gp, L, c.lane, slot_base, count);
            const bool owner = ((c.lane & (L - 1)) & ~(NVP - 1)) == 0;
#pragma unroll
            for (int i = 0; i < NVP; ++i) {
                if (i < count) {
                    const int slot = slot_base + i;
                    const int rb = slot / NG, v = slot - rb * NG;
                    const int r = gr + rb * g.rg;
                    if (owner && rb < RPT && rb < g.rpt && r < nrows) RG[((size_t)(grow0 + r) * wpr + wir) * NG + v] = gp[i];
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
    if (!hier_reduce(g, f, rec, 3, &c.ctl->flag)) return;
    if (threadIdx.x == 0) {
        const double dm = INITIAL ? part_dmax(g, f) : 0.0;
        if (a.flags & kFlagPartial) {
            f.scal[0] = rec[0]; f.scal[1] = rec[1]; f.scal[2] = rec[2]; f.scal[3] = dm;
        } else if (INITIAL) {
            state_setup(st, f, rec, dm, g, Acur);
        } else {
            state_close_outer(st, f, rec[0], a.tol);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Column ownership of a thread.  C <= 2: C adjacent columns starting at C * tc.  C == 4: two adjacent pairs 2 * ntc columns
// apart (columns 2 tc, 2 tc + 1, 2 tc + 2 ntc, 2 tc + 2 ntc + 1), so that every vector load of a warp is contiguous in shared
// memory (no bank conflicts) and even row pitches suffice.  Pairs beyond N are redirected to column 0: they read valid data,
// their alpha entries are zero and their results are never stored.
template <int C>
__device__ __forceinline__ int col_index(int tc, int ntc, int cc) { return C == 4 ? 2 * tc + (cc & 1) + (cc >> 1) * 2 * ntc : C * tc + cc; }

template <typename T, typename WT, int C>
struct ColLoader {
    static constexpr int NP = C == 4 ? 2 : 1;
    unsigned xo[NP], dofs[NP];
    bool pvalid[NP];
    __device__ __forceinline__ void init(const Geom& g, int tc) {
#pragma unroll
        for (int p = 0; p < NP; ++p) {
            const int jb = col_index<C>(tc, g.ntc, 2 * p);
            pvalid[p] = jb < g.N;
            const int j = pvalid[p] ? jb : 0;
            xo[p] = g.offX + (unsigned)(j * sizeof(T));
            dofs[p] = g.offD + (unsigned)(j * sizeof(WT));
        }
    }
    // rx / rd: byte offset of the row inside the X / D region of the stage
    __device__ __forceinline__ void load(uint32_t sb, unsigned rx, unsigned rd, T (&x)[C], T (&d)[C]) const {
        if (C == 4) {
#pragma unroll
            for (int p = 0; p < NP; ++p) {
                T xx[2], dd[2];
                lds2(sb + xo[p] + rx, xx[0], xx[1]);
                WLoad<T, WT, 2>::ld(sb + dofs[p] + rd, dd);
                x[(2 * p) % C] = xx[0]; x[(2 * p + 1) % C] = xx[1];
                d[(2 * p) % C] = dd[0]; d[(2 * p + 1) % C] = dd[1];
            }
        } else {
            ldsC<T, C>(sb + xo[0] + rx, x);
            WLoad<T, WT, C>::ld(sb + dofs[0] + rd, d);
        }
    }
};

// ------------------------------------------------------------------------------------------------
// rowgram pass, 4 columns per thread (two pairs, see ColLoader).  Differences to rowgram_kernel:
//  * a thread owns 4 adjacent columns and RPT rows of the tile -> the broadcast [R_trunc | u] row loads, the address
//    arithmetic and the per-tile ring bookkeeping are spread over 4 x RPT elements;
//  * the row -> register-slot assignment is lane dependent (slot rb holds tile row rb ^ rmask(lane)), so the first
//    log2(RPT) butterfly steps need no selects: every lane keeps its low slots and sends its high slots;
//  * the cost is assembled from  sum d c^2  (one FMA per element, per-thread accumulator) and the row statistics:
//    sum_j d (c - u a_u)^2 = sum_j d c^2 - 2 u^T b + u^T H u  (writer lanes add the last two terms per row).
template <typename T, typename WT, int KB, int NUB, int RPT, bool INITIAL>
__global__ void __launch_bounds__(kThreads, rowgram_min_blocks(KB, NUB, 4, RPT)) rowgram4_kernel(const PassArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int C = 4;
    constexpr int NG = ng_of(NUB);
    constexpr int LOGR = RPT == 4 ? 2 : (RPT == 2 ? 1 : 0);
    static_assert(RPT == 1 || RPT == 2 || RPT == 4, "RPT must be 1, 2 or 4");
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
    constexpr int NSRC = 5;
    const bool multmode = g.multmode != 0;       // bootstrap resample in multiplicity form: rows are source rows, weighted by mult
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(T), g.offX, 1, (unsigned char)(g.row_bulk & 1u), 0};
        src[1] = {f.D, g.ldd * (long long)sizeof(WT), g.offD, 1, (unsigned char)((g.row_bulk >> 1) & 1u), 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(T), g.offR, 1, (unsigned char)((g.row_bulk >> 2) & 1u), 0};
        src[3] = {multmode ? nullptr : Ucur, g.ldu * (long long)sizeof(T), g.offU, 0, 0, 0};
        src[4] = {multmode ? reinterpret_cast<const char*>(f.mult) : nullptr, 4, g.offUp, 0, 0, 0};
    }
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, NSRC);
    {
        const int tc = c.ctid % g.ntc, gr = c.ctid / g.ntc;
        ColLoader<T, WT, C> cl;
        cl.init(g, tc);
        const int L = min(g.ntc, 32);
        const int wpr = (g.ntc + 31) / 32;
        const int wir = tc >> 5;
        int rmask = 0, nsplit = 0;
#pragma unroll
        for (int s = 0; s < LOGR; ++s)
            if ((1 << s) < L) {
                ++nsplit;
                if ((c.lane >> s) & 1) rmask |= 1 << (LOGR - 1 - s);
            }
        const int nslots = RPT >> nsplit;
        const bool writer = ((c.lane & (L - 1)) >> nsplit) == 0;
        T ak[KB > 0 ? KB : 1][C];
        T au[NUB][C];
#pragma unroll
        for (int k = 0; k < KB; ++k)
#pragma unroll
            for (int cc = 0; cc < C; ++cc) {
                const int j = col_index<C>(tc, g.ntc, cc);
                ak[k][cc] = (k < g.K && j < g.N) ? Acur[(size_t)k * g.N + j] : (T)0;
            }
#pragma unroll
        for (int q = 0; q < NUB; ++q)
#pragma unroll
            for (int cc = 0; cc < C; ++cc) {
                const int j = col_index<C>(tc, g.ntc, cc);
                au[q][cc] = (q < g.nu && j < g.N) ? Acur[(size_t)(g.K + q) * g.N + j] : (T)0;
            }
        const unsigned xpitch = (unsigned)(g.ldx * sizeof(T)), dpitch = (unsigned)(g.ldd * sizeof(WT));
        const unsigned rpitch = (unsigned)(g.ldr * sizeof(T)), upitch = (unsigned)(g.ldu * sizeof(T));
        const int nRch = g.Kp >> 1, nUch = g.nup >> 1;
        double* RG = f.rowgram;
        // A tile holds g.rpt rows per row group, processed in batches of RPT (g.rpt is a multiple of RPT, or smaller than RPT: then
        // the slots beyond it are dead).  Per-slot constants (the same for every tile and batch): tile row of the slot within
        // batch 0 and its byte offsets in the X, D, R, U regions.  Dead slots alias slot 0's row; rows beyond the end of the last
        // tile read stale rows of the stage: neither is ever stored or counted.
        int rowi[RPT];
        unsigned ox[RPT], od[RPT], orr[RPT], ou[RPT];
#pragma unroll
        for (int rb = 0; rb < RPT; ++rb) {
            const int rl = rb ^ rmask;
            const int rowe = gr + (rl < g.rpt ? rl : 0) * g.rg;
            rowi[rb] = rl < g.rpt ? rowe : 0x3fffffff;
            ox[rb] = rowe * xpitch; od[rb] = rowe * dpitch; orr[rb] = g.offR + rowe * rpitch; ou[rb] = g.offU + rowe * upitch;
        }
        unsigned rco[KB > 1 ? KB / 2 : 1], uco[(NUB + 1) / 2];
#pragma unroll
        for (int i = 0; i < KB / 2; ++i) rco[i] = (i < nRch ? i : 0) * 2 * (unsigned)sizeof(T);
#pragma unroll
        for (int i = 0; i < (NUB + 1) / 2; ++i) uco[i] = (i < nUch ? i : 0) * 2 * (unsigned)sizeof(T);
        // au (x) au per owned column (few unknown types only: registers): H_m = sum_j d_mj P_j
        constexpr bool USE_P = NUB <= 2;
        T P[USE_P ? NG - NUB : 1][C];
        if (USE_P) {
#pragma unroll
            for (int q = 0; q < NUB; ++q)
#pragma unroll
                for (int q2 = q; q2 < NUB; ++q2)
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) P[USE_P ? tri_index(q, q2, NUB) : 0][cc] = au[q][cc] * au[q2][cc];
        }
        const int nbatch = g.rpt > RPT ? g.rpt / RPT : 1;
        const unsigned bx = (unsigned)(RPT * g.rg) * xpitch, bd = (unsigned)(RPT * g.rg) * dpitch, br = (unsigned)(RPT * g.rg) * rpitch,
                       bu = (unsigned)(RPT * g.rg) * upitch;

        for (; cr.it < c.n_my; cr.advance(g, stages32)) {
            produce_next(g, f, c, pr, stages32, NSRC);
            mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
            const uint32_t sb = cr.sb;
            const int nrows = cr.rows(g, c);
            const long long grow0 = (long long)cr.gtile * g.tile_rows;

          for (int bb = 0; bb < nbatch; ++bb) {
            const int brow = bb * RPT * g.rg;                      // first tile row of the batch (row group 0, slot row 0)
            const uint32_t sbx = sb + bb * bx, sbd = sb + bb * bd, sbr = sb + bb * br, sbu = sb + bb * bu;
            double gp[RPT][NG];
#pragma unroll
            for (int rb = 0; rb < RPT; ++rb) {
                const bool live = rowi[rb] + brow < nrows;
                T rk[KB > 0 ? KB : 1], uc[NUB > 1 ? NUB : 2];
#pragma unroll
                for (int i = 0; i < KB / 2; ++i) lds2(sbr + orr[rb] + rco[i], rk[2 * i], rk[2 * i + 1]);
                if (!multmode) {
#pragma unroll
                    for (int i = 0; i < (NUB + 1) / 2; ++i) lds2(sbu + ou[rb] + uco[i], uc[2 * i], uc[2 * i + 1]);
                }
                double wrow = 1.0;                                 // multiplicity of the row (1 outside multiplicity form)
                if (multmode) {
                    int mlt;
                    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(mlt) : "r"(sb + g.offUp + 4u * (unsigned)(live ? rowi[rb] + brow : 0)));
                    wrow = (double)mlt;
                }
                if (INITIAL && tc == 0 && live) {
                    double sr = 0.0;
#pragma unroll
                    for (int k = 0; k < KB; ++k)
                        if (k < g.K) sr = fma((double)rk[k], (double)rk[k], sr);
                    ssq_r = fma(wrow, sr, ssq_r);
                    if (!multmode) {
#pragma unroll
                        for (int q = 0; q < NUB; ++q)
                            if (q < g.nu) ssq_u = fma((double)uc[q], (double)uc[q], ssq_u);
                    }
                }
                T x[C], d[C], cres[C], z[C];
                cl.load(sb, bb * bx + ox[rb], bb * bd + od[rb], x, d);
                if (INITIAL && live && wrow > 0.0) {
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) dmx = fmax(dmx, (double)d[cc]);
                }
                if (KB > 0) {
                    T pk[C], pk1[C];
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) { pk[cc] = rk[0] * ak[0][cc]; pk1[cc] = rk[KB > 1 ? 1 : 0] * ak[KB > 1 ? 1 : 0][cc]; }
#pragma unroll
                    for (int k = 2; k < KB; k += 2)
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) {
                            pk[cc] = fma_t<T>(rk[k], ak[k][cc], pk[cc]);
                            pk1[cc] = fma_t<T>(rk[k + 1], ak[k + 1][cc], pk1[cc]);
                        }
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) cres[cc] = x[cc] - (pk[cc] + pk1[cc]);     // c = x - R_trunc a_k
                } else {
#pragma unroll
                    for (int cc = 0; cc < C; ++cc) cres[cc] = x[cc];
                }
#pragma unroll
                for (int cc = 0; cc < C; ++cc) z[cc] = d[cc] * cres[cc];
                {
                    const T ccA = fma_t<T>(z[1], cres[1], z[0] * cres[0]), ccB = fma_t<T>(z[3], cres[3], z[2] * cres[2]);
                    if (live) cost = fma(wrow, (cl.pvalid[0] ? (double)ccA : 0.0) + (cl.pvalid[1] ? (double)ccB : 0.0), cost);
                }
#pragma unroll
                for (int q = 0; q < NUB; ++q) {
                    T bq = z[0] * au[q][0];
#pragma unroll
                    for (int cc = 1; cc < C; ++cc) bq = fma_t<T>(z[cc], au[q][cc], bq);
                    gp[rb][q] = (double)bq;
                }
                if (USE_P) {
#pragma unroll
                    for (int e = 0; e < NG - NUB; ++e) {
                        T h = d[0] * P[USE_P ? e : 0][0];
#pragma unroll
                        for (int cc = 1; cc < C; ++cc) h = fma_t<T>(d[cc], P[USE_P ? e : 0][cc], h);
                        gp[rb][NUB + e] = (double)h;
                    }
                } else {
#pragma unroll
                    for (int q = 0; q < NUB; ++q) {
                        T t[C];
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) t[cc] = d[cc] * au[q][cc];
#pragma unroll
                        for (int q2 = q; q2 < NUB; ++q2) {
                            T h = t[0] * au[q2][0];
#pragma unroll
                            for (int cc = 1; cc < C; ++cc) h = fma_t<T>(t[cc], au[q2][cc], h);
                            gp[rb][NUB + tri_index(q, q2, NUB)] = (double)h;
                        }
                    }
                }
            }
            // select-free butterfly: split steps halve the slots, then plain xor steps on the remaining slot
#pragma unroll
            for (int s = 0; s < 5; ++s) {
                const int o = 1 << s;
                if (o < L) {
                    if (s < LOGR) {
                        constexpr int dummy = 0; (void)dummy;
                        const int half = RPT >> (s + 1);
#pragma unroll
                        for (int i = 0; i < RPT / 2; ++i)
                            if (i < half) {
#pragma unroll
                                for (int v = 0; v < NG; ++v) gp[i][v] += __shfl_xor_sync(0xffffffffu, gp[(i + half) % RPT][v], o);
                            }
                    } else {
#pragma unroll
                        for (int v = 0; v < NG; ++v) gp[0][v] += __shfl_xor_sync(0xffffffffu, gp[0][v], o);
                    }
                }
            }
            if (writer) {
#pragma unroll
                for (int i = 0; i < RPT; ++i) {
                    if (i < nslots) {
                        const int r = rowi[i] + brow;
                        if (r < nrows) {
                            double* dst = RG + ((size_t)(grow0 + r) * wpr + wir) * NG;
#pragma unroll
                            for (int v = 0; v < NG; ++v) dst[v] = gp[i][v];
                            if (multmode) continue;     // cross terms need the per-position u: cost_cross_kernel adds them
                            // cost cross terms of this row (per-warp partial statistics are linear, so partial rows add up)
                            T un[NUB > 1 ? NUB : 2];
#pragma unroll
                            for (int k = 0; k < (NUB + 1) / 2; ++k) {
                                const int kk = k < nUch ? k : 0;
                                lds2(sb + g.offU + kk * 2 * (unsigned)sizeof(T) + r * upitch, un[2 * k], un[2 * k + 1]);
                            }
                            double ct = 0.0;
#pragma unroll
                            for (int q = 0; q < NUB; ++q) {
                                const double uq = (q < g.nu) ? (double)un[q] : 0.0;
                                double hq = 0.0;
#pragma unroll
                                for (int q2 = 0; q2 < NUB; ++q2) {
                                    const double u2 = (q2 < g.nu) ? (double)un[q2] : 0.0;
                                    hq = fma(gp[i][NUB + (q <= q2 ? tri_index(q, q2, NUB) : tri_index(q2, q, NUB))], u2, hq);
                                }
                                ct = fma(uq, hq - 2.0 * gp[i][q], ct);
                            }
                            cost += ct;
                        }
                    }
                }
            }
          }     // batches of the tile
            __syncwarp();
            if (c.lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));
        }
    }
    __syncthreads();
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
    if (!hier_reduce(g, f, rec, 3, &c.ctl->flag)) return;
    if (threadIdx.x == 0) {
        const double dm = INITIAL ? part_dmax(g, f) : 0.0;
        if ((a.flags & kFlagPartial) || multmode) {
            f.scal[0] = rec[0]; f.scal[1] = rec[1]; f.scal[2] = rec[2]; f.scal[3] = dm;
        } else if (INITIAL) {
            state_setup(st, f, rec, dm, g, Acur);
        } else {
            state_close_outer(st, f, rec[0], a.tol);
        }
    }
}

// ------------------------------------------------------------------------------------------------
// n_iter2 iterations of update_u (deconvolution.py:82-89; gradient at u for the unsupervised variant, :163) per row,
// on the row's (b, H).  One thread per row; both U slots are rewritten (u and u_ persist across outer iterations).
template <typename T, int NUB>
__global__ void __launch_bounds__(kThreads) u_inner_kernel(const PassArgs a) {
    constexpr int NG = ng_of(NUB);
    __shared__ double scratch[16];
    __shared__ double rec[2];
    __shared__ int flag;
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    const int n2 = a.k_inner;
    const int ucur = st->u_cur;
    const double l_w = st->l_w, lwo_in = st->l_w_old;
    const T inv_lw = (T)1 / (T)l_w;      // step 1 / l_w as a reciprocal multiply: <= 1 ulp of a ~1e-4-sized step vs the division of :88
    const int t0 = st->t_u;
    const double* mm = a.mom_m + t0;
    // beta_t = min((a_t - 1) / a_{t+1}, 0.9999 sqrt(l_w_ / l_w)); l_w_ == l_w from the second inner iteration on (:89)
    const double cap0 = 0.9999 * sqrt(lwo_in / l_w), cap1 = 0.9999 * sqrt(l_w / l_w);
    T* Uc = reinterpret_cast<T*>(f.U + (size_t)ucur * g.uslot_bytes);
    T* Up = reinterpret_cast<T*>(f.U + (size_t)(ucur ^ 1) * g.uslot_bytes);
    const bool at_current = (g.mode == 2);
    const int wpr = (g.ntc + 31) / 32;
    const double* RG = f.rowgram;
    double ssq = 0.0;
    for (long long row = (long long)part_id(g) * blockDim.x + threadIdx.x; row < g.M; row += (long long)g.n_parts * blockDim.x) {
        double v[NG];
#pragma unroll
        for (int i = 0; i < NG; ++i) v[i] = 0.0;
        for (int w = 0; w < wpr; ++w) {
            const double* p = RG + ((size_t)row * wpr + w) * NG;
#pragma unroll
            for (int i = 0; i < NG; ++i) v[i] += __ldcg(p + i);
        }
        T u[NUB], up[NUB];
#pragma unroll
        for (int q = 0; q < NUB; ++q) {
            u[q] = q < g.nu ? Uc[(size_t)row * g.ldu + q] : (T)0;
            up[q] = q < g.nu ? Up[(size_t)row * g.ldu + q] : (T)0;
        }
        for (int it = 0; it < n2; ++it) {
            const T beta = (T)fmin(__ldg(mm + it), it == 0 ? cap0 : cap1);
            T ut[NUB], ug[NUB];
#pragma unroll
            for (int q = 0; q < NUB; ++q) {
                ut[q] = u[q] + beta * (u[q] - up[q]);
                ug[q] = at_current ? u[q] : ut[q];
            }
#pragma unroll
            for (int q = 0; q < NUB; ++q) {
                double s = 0.0;
#pragma unroll
                for (int q2 = 0; q2 < NUB; ++q2) {
                    const double h = v[NUB + (q <= q2 ? tri_index(q, q2, NUB) : tri_index(q2, q, NUB))];
                    s = fma(h, (double)ug[q2], s);
                }
                const double gq = v[q] - s;
                T un = ut[q] + (T)gq * inv_lw;
                un = clip01(un);
                up[q] = u[q];
                u[q] = un;
            }
        }
#pragma unroll
        for (int q = 0; q < NUB; ++q)
            if (q < g.nu) {
                Uc[(size_t)row * g.ldu + q] = u[q];
                Up[(size_t)row * g.ldu + q] = up[q];
                ssq = fma((double)u[q], (double)u[q], ssq);
            }
    }
    const double s0 = consumer_block_sum(ssq, scratch, threadIdx.x);
    if (threadIdx.x == 0) f.part[(size_t)part_id(g) * g.part_stride] = s0;
    if (!hier_reduce(g, f, rec, 1, &flag)) return;
    if (threadIdx.x == 0) {
        state_end_u(st, a.mom_a[t0 + n2], t0 + n2, l_w, n2 > 0);
        if (a.flags & kFlagPartial) f.scal[4] = rec[0];      // this GPU's rows; alpha_inner_kernel forms l_h from the all-reduced sum
        else state_u_norm(st, rec[0]);
    }
}

// ------------------------------------------------------------------------------------------------
// Multiplicity form (bootstrap resamples, bootstrap.py:28).  Position p of the resample (positions are sorted by source row,
// rows[p] = its source row) owns one row of u; all positions of a source row m share (b_m, H_m).
//   u_inner_mult_kernel : one thread per POSITION (no divergence over the multiplicities): n_iter2 update_u iterations
//   usum_kernel         : one thread per SOURCE row: usum[m] = [sum_p u_p | upper triangle of sum_p u_p u_p^T] for the Gram
//                         panel pass, which can then stream the shared, contiguous X / d_x / R_trunc instead of gathering rows
//   cost_cross_kernel   : one thread per position: the per-position terms of the cost, then the set-up / termination logic
template <typename T, int NUB>
__device__ __forceinline__ void load_rowstats(const double* RG, long long row, int wpr, double (&v)[ng_of(NUB)]) {
    constexpr int NG = ng_of(NUB);
#pragma unroll
    for (int i = 0; i < NG; ++i) v[i] = 0.0;
    for (int w = 0; w < wpr; ++w) {
        const double* p = RG + ((size_t)row * wpr + w) * NG;
#pragma unroll
        for (int i = 0; i < NG; ++i) v[i] += __ldcg(p + i);
    }
}

template <typename T, int NUB>
__global__ void __launch_bounds__(kThreads) u_inner_mult_kernel(const PassArgs a) {
    constexpr int NG = ng_of(NUB);
    __shared__ double scratch[16];
    __shared__ double rec[2];
    __shared__ int flag;
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    const int n2 = a.k_inner;
    const int ucur = st->u_cur;
    const double l_w = st->l_w, lwo_in = st->l_w_old;
    const T inv_lw = (T)1 / (T)l_w;
    const int t0 = st->t_u;
    const double* mm = a.mom_m + t0;
    const double cap0 = 0.9999 * sqrt(lwo_in / l_w), cap1 = 0.9999 * sqrt(l_w / l_w);
    T* Uc = reinterpret_cast<T*>(f.U + (size_t)ucur * g.uslot_bytes);
    T* Up = reinterpret_cast<T*>(f.U + (size_t)(ucur ^ 1) * g.uslot_bytes);
    const int wpr = (g.ntc + 31) / 32;
    double ssq = 0.0;
    for (long long pos = (long long)part_id(g) * blockDim.x + threadIdx.x; pos < g.M; pos += (long long)g.n_parts * blockDim.x) {
        double v[NG];
        load_rowstats<T, NUB>(f.rowgram, f.pos_row[pos], wpr, v);
        T u[NUB], up[NUB];
#pragma unroll
        for (int q = 0; q < NUB; ++q) {
            u[q] = q < g.nu ? Uc[(size_t)pos * g.ldu + q] : (T)0;
            up[q] = q < g.nu ? Up[(size_t)pos * g.ldu + q] : (T)0;
        }
        for (int it = 0; it < n2; ++it) {
            const T beta = (T)fmin(__ldg(mm + it), it == 0 ? cap0 : cap1);
            T ut[NUB];
#pragma unroll
            for (int q = 0; q < NUB; ++q) ut[q] = u[q] + beta * (u[q] - up[q]);
#pragma unroll
            for (int q = 0; q < NUB; ++q) {
                double sq = 0.0;
#pragma unroll
                for (int q2 = 0; q2 < NUB; ++q2)
                    sq = fma(v[NUB + (q <= q2 ? tri_index(q, q2, NUB) : tri_index(q2, q, NUB))], (double)ut[q2], sq);
                T un = ut[q] + (T)(v[q] - sq) * inv_lw;
                un = clip01(un);
                up[q] = u[q];
                u[q] = un;
            }
        }
#pragma unroll
        for (int q = 0; q < NUB; ++q)
            if (q < g.nu) {
                Uc[(size_t)pos * g.ldu + q] = u[q];
                Up[(size_t)pos * g.ldu + q] = up[q];
                ssq = fma((double)u[q], (double)u[q], ssq);
            }
    }
    const double s0 = consumer_block_sum(ssq, scratch, threadIdx.x);
    if (threadIdx.x == 0) f.part[(size_t)part_id(g) * g.part_stride] = s0;
    if (!hier_reduce(g, f, rec, 1, &flag)) return;
    if (threadIdx.x == 0) {
        state_end_u(st, a.mom_a[t0 + n2], t0 + n2, l_w, n2 > 0);
        state_u_norm(st, rec[0]);
    }
}

template <typename T, int NUB>
__global__ void __launch_bounds__(kThreads) usum_kernel(const PassArgs a) {
    constexpr int NG = ng_of(NUB);
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    if (f.st->done) return;
    const T* Uc = reinterpret_cast<const T*>(f.U + (size_t)f.st->u_cur * g.uslot_bytes);
    for (long long row = (long long)part_id(g) * blockDim.x + threadIdx.x; row < g.M; row += (long long)g.n_parts * blockDim.x) {
        const int p0 = f.offs[row], p1 = f.offs[row + 1];
        double us[NG];
#pragma unroll
        for (int i = 0; i < NG; ++i) us[i] = 0.0;
        for (int pos = p0; pos < p1; ++pos) {
            double u[NUB];
#pragma unroll
            for (int q = 0; q < NUB; ++q) u[q] = q < g.nu ? (double)Uc[(size_t)pos * g.ldu + q] : 0.0;
#pragma unroll
            for (int q = 0; q < NUB; ++q) {
                us[q] += u[q];
#pragma unroll
                for (int q2 = q; q2 < NUB; ++q2) us[NUB + tri_index(q, q2, NUB)] = fma(u[q], u[q2], us[NUB + tri_index(q, q2, NUB)]);
            }
        }
        double* dst = f.usum + (size_t)row * NG;
#pragma unroll
        for (int i = 0; i < NG; ++i) dst[i] = us[i];
    }
}

// cost of the current iterate in multiplicity form: rowgram4_kernel left  sum_m mult_m sum_j d c^2  (and ||R||^2, max d) in
// FitDev::scal; this kernel adds the per-position terms  -2 u_p^T b_m + u_p^T H_m u_p  (and ||u||^2 at set-up) and runs the
// set-up / termination logic (deconvolution.py:192-204, :218-221).
template <typename T, int NUB>
__global__ void __launch_bounds__(kThreads) cost_cross_kernel(const PassArgs a) {
    constexpr int NG = ng_of(NUB);
    __shared__ double scratch[16];
    __shared__ double rec[4];
    __shared__ int flag;
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    const bool initial = (a.flags & kFlagInitial) != 0;
    const int ucur = st->u_cur, acur = st->a_cur;
    const T* Uc = reinterpret_cast<const T*>(f.U + (size_t)ucur * g.uslot_bytes);
    const int wpr = (g.ntc + 31) / 32;
    double cross = 0.0, ssq = 0.0;
    for (long long pos = (long long)part_id(g) * blockDim.x + threadIdx.x; pos < g.M; pos += (long long)g.n_parts * blockDim.x) {
        double v[NG];
        load_rowstats<T, NUB>(f.rowgram, f.pos_row[pos], wpr, v);
        double u[NUB];
#pragma unroll
        for (int q = 0; q < NUB; ++q) u[q] = q < g.nu ? (double)Uc[(size_t)pos * g.ldu + q] : 0.0;
        double ct = 0.0;
#pragma unroll
        for (int q = 0; q < NUB; ++q) {
            double hq = 0.0;
#pragma unroll
            for (int q2 = 0; q2 < NUB; ++q2) hq = fma(v[NUB + (q <= q2 ? tri_index(q, q2, NUB) : tri_index(q2, q, NUB))], u[q2], hq);
            ct = fma(u[q], hq - 2.0 * v[q], ct);
            ssq = fma(u[q], u[q], ssq);
        }
        cross += ct;
    }
    const double s0 = consumer_block_sum(cross, scratch, threadIdx.x);
    const double s1 = consumer_block_sum(ssq, scratch, threadIdx.x);
    if (threadIdx.x == 0) {
        double* p = f.part + (size_t)part_id(g) * g.part_stride;
        p[0] = s0; p[1] = s1;
    }
    if (!hier_reduce(g, f, rec, 2, &flag)) return;
    if (threadIdx.x == 0) {
        const double r4[4] = {f.scal[0] + rec[0], f.scal[1], rec[1], f.scal[3]};
        const T* Acur = reinterpret_cast<const T*>(f.A + (size_t)acur * g.Kt * g.N * sizeof(T));
        if (initial) state_setup(st, f, r4, r4[3], g, Acur);
        else state_close_outer(st, f, r4[0], a.tol);
    }
}

// ------------------------------------------------------------------------------------------------
// Per-sample Gram panel:  acc[p][q][j] = sum_m d_mj za_p(m) zb_q(m),  accx[p][j] = sum_m d_mj za_p(m) x_mj
// za = PA consecutive entries of the padded register row [R_trunc (Kp) | u (nup)] starting at chunk a.ca0 (chunks of two),
// zb = PB entries starting at chunk a.cb0.  The last CTA scatters the totals (and their mirror images) into
// gram[Kt][Kt][N] and, when a.with_x, gbx[Kt][N].
template <typename T, typename WT, int PA, int PB, int C, bool MULT>
__global__ void __launch_bounds__(kThreads, panel_min_blocks(PA, PB, C)) gram_panel_kernel(const PassArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    constexpr int NA = PA / 2, NB = PB / 2;      // PA == 1 (NA == 0) exists for the MULT u block with a single unknown type only
    static_assert(PA >= 2 || MULT, "PA = 1 is a multiplicity-form instantiation");
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    CtaCtx c;
    cta_setup(g, smem, c);
    unsigned char* stages = smem + kCtlBytes;
    const uint32_t stages32 = smem_u32(stages);
    const int ucur = st->u_cur;
    const char* Ucur = f.U + (size_t)ucur * g.uslot_bytes;
    const int tc = c.ctid % g.ntc, gr = c.ctid / g.ntc;
    const bool colvalid = col_index<C>(tc, g.ntc, 0) < g.N;      // the first owned column (C == 4: first pair) exists
    double acc[PA][PB][C], accx[PA][C];
#pragma unroll
    for (int p = 0; p < PA; ++p)
#pragma unroll
        for (int cc = 0; cc < C; ++cc) {
            accx[p][cc] = 0.0;
#pragma unroll
            for (int q = 0; q < PB; ++q) acc[p][q][cc] = 0.0;
        }
    constexpr int NSRC = MULT ? 5 : 4;
    const int nub = a.k_inner;                       // MULT: unknown-type bucket of the usum records (NG = ng_of(nub) doubles per row)
    const unsigned uspitch = (unsigned)(ng_of(nub) * 8);
    if (threadIdx.x == 0) {
        TileSrc* src = c.ctl->src;
        src[0] = {f.X, g.ldx * (long long)sizeof(T), g.offX, 1, (unsigned char)(g.row_bulk & 1u), 0};
        src[1] = {f.D, g.ldd * (long long)sizeof(WT), g.offD, 1, (unsigned char)((g.row_bulk >> 1) & 1u), 0};
        src[2] = {g.K ? f.Rk : nullptr, g.ldr * (long long)sizeof(T), g.offR, 1, (unsigned char)((g.row_bulk >> 2) & 1u), 0};
        if (MULT) {
            // multiplicity form: the u block reads the per-source-row sums usum, the known block the multiplicities
            const bool a_is_u = a.ca0 >= (g.Kp >> 1);
            src[3] = {a_is_u ? reinterpret_cast<const char*>(f.usum) : nullptr, (long long)uspitch, g.offU, 0, 0, 0};
            src[4] = {a_is_u ? nullptr : reinterpret_cast<const char*>(f.mult), 4, g.offUp, 0, 0, 0};
        } else {
            src[3] = {Ucur, g.ldu * (long long)sizeof(T), g.offU, 0, 0, 0};
        }
    }
    __syncthreads();
    Ring pr, cr;
    pr.init(g, stages32);
    cr.init(g, stages32);
    for (int i = 0; i < n_stages(g) - 2; ++i) produce_next(g, f, c, pr, stages32, NSRC);
    const int nR = g.Kp >> 1, nU = g.nup >> 1;
    {
        // chunk -> (offset, pitch) inside a stage; chunks beyond the row alias chunk 0 (their totals are dropped)
        unsigned aoff[NA > 0 ? NA : 1], apitch[NA > 0 ? NA : 1], boff[NB], bpitch[NB];
        auto locate = [&](int ch, unsigned& off, unsigned& pitch) {
            if (ch >= nR + nU) ch = 0;
            if (ch < nR) { off = g.offR + ch * 2 * (unsigned)sizeof(T); pitch = (unsigned)(g.ldr * sizeof(T)); }
            else { off = g.offU + (ch - nR) * 2 * (unsigned)sizeof(T); pitch = (unsigned)(g.ldu * sizeof(T)); }
        };
#pragma unroll
        for (int i = 0; i < NA; ++i) locate(a.ca0 + i, aoff[i], apitch[i]);
#pragma unroll
        for (int i = 0; i < NB; ++i) locate(a.cb0 + i, boff[i], bpitch[i]);
        const unsigned xpitch = (unsigned)(g.ldx * sizeof(T)), dpitch = (unsigned)(g.ldd * sizeof(WT));
        ColLoader<T, WT, C> cl;
        cl.init(g, tc);
        for (; cr.it < c.n_my; cr.advance(g, stages32)) {
            produce_next(g, f, c, pr, stages32, NSRC);
            mbar_wait(smem_u32(&c.ctl->full[cr.s]), cr.parity);
            const uint32_t sb = cr.sb;
            const int nrows = cr.rows(g, c);
            if (MULT) {
                if (colvalid) {
                    const bool a_is_u = a.ca0 >= nR;
                    for (int r = gr; r < nrows; r += g.rg) {
                        T x[C], d[C];
                        cl.load(sb, r * xpitch, r * dpitch, x, d);
                        double zax[PA], w[PA][PB];
                        if (a_is_u) {
#pragma unroll
                            for (int p = 0; p < PA; ++p) {
                                const int q = 2 * (a.ca0 - nR) + p;
                                zax[p] = 0.0;
                                if (q < nub) lds1(sb + g.offU + r * uspitch + 8u * (unsigned)q, zax[p]);
                            }
                        } else {
                            int mlt;
                            asm volatile("ld.shared.s32 %0, [%1];" : "=r"(mlt) : "r"(sb + g.offUp + 4u * (unsigned)r));
                            T za[PA >= 2 ? PA : 2];
#pragma unroll
                            for (int i = 0; i < NA; ++i) lds2(sb + aoff[i] + r * apitch[i], za[2 * i], za[2 * i + 1]);
#pragma unroll
                            for (int p = 0; p < PA; ++p) zax[p] = PA >= 2 ? (double)mlt * (double)za[p] : 0.0;
                        }
#pragma unroll
                        for (int i = 0; i < NB; ++i) {
                            const int ch = a.cb0 + i;
                            if (ch < nR) {
                                T z0, z1;
                                lds2(sb + boff[i] + r * bpitch[i], z0, z1);
#pragma unroll
                                for (int p = 0; p < PA; ++p) { w[p][2 * i] = zax[p] * (double)z0; w[p][2 * i + 1] = zax[p] * (double)z1; }
                            } else {
#pragma unroll
                                for (int p = 0; p < PA; ++p)
#pragma unroll
                                    for (int e = 0; e < 2; ++e) {
                                        const int qa = 2 * (a.ca0 - nR) + p, qb = 2 * (ch - nR) + e;
                                        double sv = 0.0;
                                        if (a_is_u && ch < nR + nU && qa < nub && qb < nub) {
                                            const int lo = qa < qb ? qa : qb, hi = qa < qb ? qb : qa;
                                            lds1(sb + g.offU + r * uspitch + 8u * (unsigned)(nub + tri_index(lo, hi, nub)), sv);
                                        }
                                        w[p][2 * i + e] = sv;
                                    }
                            }
                        }
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) {
                            const double dd = (double)d[cc], dx = dd * (double)x[cc];
#pragma unroll
                            for (int p = 0; p < PA; ++p) {
                                accx[p][cc] = fma(dx, zax[p], accx[p][cc]);
#pragma unroll
                                for (int q = 0; q < PB; ++q) acc[p][q][cc] = fma(dd, w[p][q], acc[p][q][cc]);
                            }
                        }
                    }
                }
            } else if (colvalid) {
                for (int r = gr; r < nrows; r += g.rg) {
                    T za[PA >= 2 ? PA : 2], zb[PB], x[C], d[C];
#pragma unroll
                    for (int i = 0; i < NA; ++i) lds2(sb + aoff[i] + r * apitch[i], za[2 * i], za[2 * i + 1]);
#pragma unroll
                    for (int i = 0; i < NB; ++i) lds2(sb + boff[i] + r * bpitch[i], zb[2 * i], zb[2 * i + 1]);
                    cl.load(sb, r * xpitch, r * dpitch, x, d);
#pragma unroll
                    for (int p = 0; p < PA; ++p)
#pragma unroll
                        for (int cc = 0; cc < C; ++cc) {
                            const double t = (double)d[cc] * (double)za[p];
                            accx[p][cc] = fma(t, (double)x[cc], accx[p][cc]);
#pragma unroll
                            for (int q = 0; q < PB; ++q) acc[p][q][cc] = fma(t, (double)zb[q], acc[p][q][cc]);
                        }
                }
            }
            __syncwarp();
            if (c.lane == 0) mbar_arrive(smem_u32(&c.ctl->empty[cr.s]));
        }
    }
    __syncthreads();
    // CTA partial record [p][q (PB + 1, last = x)][N]: row groups are combined in fixed order, one p at a time
    double* scratch = reinterpret_cast<double*>(stages);
    double* part = f.part + (size_t)part_id(g) * g.part_stride;
    const int QN = (PB + 1) * g.N;
#pragma unroll
    for (int p = 0; p < PA; ++p) {
        for (int gg = 0; gg < g.rg; ++gg) {
            if (gr == gg && colvalid) {
#pragma unroll
                for (int cc = 0; cc < C; ++cc) {
                    const int j = col_index<C>(tc, g.ntc, cc);
                    if (j < g.N) {
#pragma unroll
                        for (int q = 0; q < PB; ++q) {
                            double* ptr = &scratch[(size_t)q * g.N + j];
                            *ptr = (gg == 0) ? acc[p][q][cc] : (*ptr + acc[p][q][cc]);
                        }
                        double* ptr = &scratch[(size_t)PB * g.N + j];
                        *ptr = (gg == 0) ? accx[p][cc] : (*ptr + accx[p][cc]);
                    }
                }
            }
            __syncthreads();
        }
        for (int e = threadIdx.x; e < QN; e += blockDim.x) part[(size_t)p * QN + e] = scratch[e];
        __syncthreads();
    }
    const int n = PA * QN;
    if (!hier_reduce(g, f, f.red, n, &c.ctl->flag)) return;
    __threadfence();
    __syncthreads();
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const int p = e / QN, rem = e - p * QN;
        const int q = rem / g.N, j = rem - q * g.N;
        const int ia = alpha_row_of(g, 2 * a.ca0 + p);
        if (ia < 0) continue;
        const double v = f.red[e];
        if (q == PB) {
            if (a.with_x) f.gbx[(size_t)ia * g.N + j] = v;
        } else {
            const int ib = alpha_row_of(g, 2 * a.cb0 + q);
            if (ib < 0) continue;
            // a diagonal launch holds (ia, ib) twice, as (p, q) and as (q', p'), computed as (d z_a) z_b and (d z_b) z_a: the two
            // roundings differ and both would be stored to the same two entries by different threads - keep the (ia <= ib) one
            const int ra = 2 * a.ca0 + p, rb = 2 * a.cb0 + q;
            if (ra > rb && rb >= 2 * a.ca0 && rb < 2 * a.ca0 + PA && ra >= 2 * a.cb0 && ra < 2 * a.cb0 + PB) continue;
            f.gram[((size_t)ia * g.Kt + ib) * g.N + j] = v;
            f.gram[((size_t)ib * g.Kt + ia) * g.N + j] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------------
// projection_simplex_sort_2d (deconvolution.py:21-37) of one column held in registers: bitonic sorting network
// (compile-time indices only), entries k >= p are padding.  Returns false when v holds a NaN (the reference
// raises ZeroDivisionError there: rho stays -1).
template <int KTB>
__device__ __forceinline__ bool project_simplex_reg(double (&v)[KTB], int p) {
    double u[KTB];
    bool nan = false;
#pragma unroll
    for (int k = 0; k < KTB; ++k) {
        u[k] = k < p ? v[k] : -1.0e300;
        nan |= (k < p) && !(v[k] == v[k]);
    }
    if (nan) return false;
#pragma unroll
    for (int kk = 2; kk <= KTB; kk <<= 1)
#pragma unroll
        for (int j = kk >> 1; j > 0; j >>= 1)
#pragma unroll
            for (int i = 0; i < KTB; ++i) {
                const int l = i ^ j;
                if (l > i) {
                    const bool desc = (i & kk) == 0;
                    // NaNs were excluded above: one comparison and selects instead of the NaN-aware fmax / fmin pair
                    const bool gt = u[i] > u[l];
                    const double hi = gt ? u[i] : u[l], lo = gt ? u[l] : u[i];
                    u[i] = desc ? hi : lo;
                    u[l] = desc ? lo : hi;
                }
            }
    double cs = 0.0, theta = 0.0;
    bool found = false;
#pragma unroll
    for (int j = 0; j < KTB; ++j) {
        if (j < p) {
            cs += u[j];
            const double pi = cs - 1.0;
            const double th = pi / (double)(j + 1);
            if (u[j] - th > 0.0) { found = true; theta = th; }
        }
    }
    if (!found) return false;
#pragma unroll
    for (int k = 0; k < KTB; ++k) { const double w = v[k] - theta; v[k] = w > 0.0 ? w : 0.0; }      // np.maximum(v - theta, 0), no NaN here
    return true;
}

// ------------------------------------------------------------------------------------------------
// projection_simplex_sort_2d (deconvolution.py:21-37) of one column spread over the L lanes of a lane group (lane k holds v[k];
// entries k >= p are padding): bitonic sort by lane exchanges, the cumulative sum in the reference's left-to-right order (one
// shuffle per step), every lane divides for its own candidate threshold, the LAST lane that satisfies the condition supplies theta.
// Same arithmetic as project_simplex_reg, value for value.  Returns false (for the whole group) when v holds a NaN.
template <int L>
__device__ __forceinline__ bool project_simplex_lanes(double& v, int k, int p, int base, double rk) {
    constexpr unsigned kFull = 0xffffffffu;
    const unsigned gsel = L == 32 ? kFull : ((1u << (L & 31)) - 1u);
    const unsigned nanb = (__ballot_sync(kFull, (k < p) && !(v == v)) >> base) & gsel;
    double u = k < p ? v : -1.0e300;
#pragma unroll
    for (int kk = 2; kk <= L; kk <<= 1)
#pragma unroll
        for (int j = kk >> 1; j > 0; j >>= 1) {
            const double o = __shfl_xor_sync(kFull, u, j, L);
            const bool desc = (k & kk) == 0, lower = (k & j) == 0;
            const bool gt = u > o;
            const double hi = gt ? u : o, lo = gt ? o : u;
            u = (lower == desc) ? hi : lo;
        }
    // cs[k] = ((u[0] + u[1]) + ...) + u[k], the reference's left-to-right order: every lane adds its own prefix (the shuffles are
    // independent of the chain of additions)
    double cs = __shfl_sync(kFull, u, 0, L);
    for (int l = 1; l < p; ++l) {
        const double t = __shfl_sync(kFull, u, l, L);
        if (l <= k) cs += t;
    }
    // (cs - 1) / (k + 1), correctly rounded without the division sequence: rk = RN(1 / (k + 1)), q0 = RN(x rk) is faithful, the FMA
    // remainder is exact and RN(q0 + rem rk) is the rounded quotient (Markstein); |x| is O(1) here, never subnormal or huge
    const double x = cs - 1.0, q0 = x * rk;
    const double th = fma(fma(-(double)(k + 1), q0, x), rk, q0);
    const unsigned condb = (__ballot_sync(kFull, (k < p) && (u - th > 0.0)) >> base) & gsel;
    const int last = condb ? 31 - __clz(condb) : 0;
    const double theta = __shfl_sync(kFull, th, last, L);
    if (nanb || !condb) return false;
    const double w = v - theta;
    v = w > 0.0 ? w : 0.0;                           // np.maximum(v - theta, 0), no NaN here
    return true;
}

// first index of the minimum of g over the lanes lo <= k < hi of a lane group, with the scan semantics of the reference's
// np.argmin on a slice that may hold NaNs restated as in the per-thread loop: the first entry is taken as it is, later entries
// replace it only if they compare smaller
template <int L>
__device__ __forceinline__ int first_argmin_lanes(double gk, int k, int lo, int hi) {
    constexpr unsigned kFull = 0xffffffffu;
    const bool in = k >= lo && k < hi;
    const int first_nan = __shfl_sync(kFull, (int)!(gk == gk), lo < L ? lo : 0, L);
    double val = (in && gk == gk) ? gk : __longlong_as_double(0x7ff0000000000000ll);
    int idx = in ? k : L;
#pragma unroll
    for (int off = L >> 1; off > 0; off >>= 1) {
        const double ov = __shfl_xor_sync(kFull, val, off, L);
        const int oi = __shfl_xor_sync(kFull, idx, off, L);
        if (ov < val || (ov == val && oi < idx)) { val = ov; idx = oi; }
    }
    return (first_nan || idx >= L) ? lo : idx;
}

// ------------------------------------------------------------------------------------------------
// n_iter2 iterations of update_alpha (deconvolution.py:94-101 with projection :21-37) or of frank_wolfe_nmf (:285-299)
// per sample column on (G_j, bx_j).  alpha and alpha_ both persist.
// The iterations of a sample are one dependent chain (extrapolation -> Kt x Kt matrix-vector product -> sort -> cumulative sum ->
// threshold), so a sample is spread over L = KTB lanes: lane k holds row k of G_j, b[k], alpha[k]; alpha_t travels by shuffles, the
// projection runs across the lanes (project_simplex_lanes).  Every value is computed by the same operations in the same order as
// with one thread per sample (the kernel this replaces: 0.041 ms per launch at N = 256, Kt = 8); the chain per iteration is ~6x shorter.
template <typename T, int KTB>
__global__ void __launch_bounds__(32) alpha_inner_kernel(const PassArgs a) {
    // grid = (fits, ceil(N / (32 / L))): a CTA is ONE warp that owns 32 / L consecutive samples, so that the samples of a fit spread
    // over many SMs (the iterations are FP64-latency bound).  The last CTA of a fit sums the per-sample ||alpha_unk||^2 in
    // sample order and updates the state; no other CTA writes it.
    constexpr int L = KTB, SPW = 32 / L;
    constexpr unsigned kFull = 0xffffffffu;
    __shared__ int s_last;
    const Geom& g = a.g;
    const FitDev f = a.fits[blockIdx.x];
    FitState* st = f.st;
    if (st->done) return;
    const bool fw = (a.flags & kFlagFW) != 0;
    const int n2 = a.k_inner, Kt = g.Kt;
    const int acur = st->a_cur;
    const bool sharded = (a.flags & kFlagPartial) != 0;
    // row-sharded: ||u||^2 summed over all GPUs -> l_h, deconvolution.py:212
    const double l_h = sharded ? lipschitz(st->ssq_rk + f.rscal[4], st->dmax2) : st->l_h;
    // Row-sharded fused engine: the fused pass published this GPU's cost / ||u||^2 / panel; on the all-reduced copies every CTA
    // takes the same termination decision (deconvolution.py:218-221), the last CTA commits it (dmf_fused.cuh, last-CTA logic)
    const bool fcommit = (a.flags & kFlagFusedCommit) != 0;
    const int phase_in = st->phase;
    const double cf_new = fcommit ? f.rscal[0] : 0.0;
    const bool fstop = fcommit && phase_in == 1 && outer_stops(cf_new, st->cf, a.tol);
    const double lw_pass = st->l_w;                      // the l_w the fused pass stepped with
    const int tu_in = st->t_u, ucur_in = st->u_cur;
    const double lho_in = st->l_h_old;
    const int t0 = st->t_a;
    const double* mm = a.mom_m + t0;
    const double cap0 = 0.9999 * sqrt(lho_in / l_h), cap1 = 0.9999 * sqrt(l_h / l_h);
    const double inv_lh = 1.0 / l_h;
    T* Acur = reinterpret_cast<T*>(f.A) + (size_t)acur * g.Kt * g.N;
    T* Aprev = reinterpret_cast<T*>(f.A) + (size_t)(acur ^ 1) * g.Kt * g.N;
    int any_bad = 0;
    const int n_cta = gridDim.y;
    {
        const int lane = threadIdx.x, k = lane % L, base = lane - k;
        const int j = blockIdx.y * SPW + lane / L;
        const bool act = j < g.N && !fstop;                  // the same for the L lanes of a sample
        const bool mine = act && k < Kt;
        double Grow[KTB];
#pragma unroll
        for (int l = 0; l < KTB; ++l) Grow[l] = (mine && l < Kt) ? f.rgram[((size_t)k * Kt + l) * g.N + j] : 0.0;
        const double b = mine ? f.rgbx[(size_t)k * g.N + j] : 0.0;
        double ac = mine ? (double)Acur[(size_t)k * g.N + j] : 0.0;
        double ap = mine ? (double)Aprev[(size_t)k * g.N + j] : 0.0;
        const double rk = 1.0 / (double)(k + 1);            // for the thresholds of the projection (one IEEE division per launch)
        if (!fw) {
            bool bad = false;                                // per sample: the iterate stays where the NaN appeared
            for (int it = 0; it < n2; ++it) {
                const double beta = (double)(T)fmin(__ldg(mm + it), it == 0 ? cap0 : cap1);
                const double at = (double)(T)(ac + beta * (ac - ap));
                double s = 0.0;
#pragma unroll
                for (int l = 0; l < KTB; ++l) s = fma(Grow[l], __shfl_sync(kFull, at, l, L), s);
                double v = (double)(T)(at + (double)(T)((b - s) * inv_lh));
                const bool ok = project_simplex_lanes<L>(v, k, Kt, base, rk);
                if (!ok) bad = true;
                if (!bad) { ap = ac; ac = k < Kt ? (double)(T)v : 0.0; }
                if (__all_sync(kFull, bad || !act)) break;
            }
            if (bad && act) any_bad = 1;
        } else {
            const double pj = act ? f.purity[j] : 0.0;
            for (int it = 0; it < n2; ++it) {
                const double gamma = 2.0 / (double)(it + 2);
                double s = 0.0;
#pragma unroll
                for (int l = 0; l < KTB; ++l) s = fma(Grow[l], __shfl_sync(kFull, ac, l, L), s);
                const double gk = -(b - s);                   // gradient, deconvolution.py:286-287
                const int i1 = first_argmin_lanes<L>(gk, k, 0, g.K);
                const int i2 = first_argmin_lanes<L>(gk, k, g.K, Kt);
                if (k < Kt) {
                    const double sv = (k < g.K) ? ((k == i1) ? pj : 0.0) : ((k == i2) ? (1.0 - pj) : 0.0);
                    ac = (double)(T)((1.0 - gamma) * ac + gamma * sv);
                }
            }
        }
        if (mine) {
            Acur[(size_t)k * g.N + j] = (T)ac;
            if (!fw) Aprev[(size_t)k * g.N + j] = (T)ap;
        }
        double sa = 0.0;                                     // ||alpha_unk[:, j]||^2 in row order
        for (int l = g.K; l < Kt; ++l) {
            const double t = __shfl_sync(kFull, ac, l, L);
            sa = fma(t, t, sa);
        }
        if (act && k == 0) f.part[j] = sa;
    }
    any_bad = __syncthreads_or(any_bad);
    if (threadIdx.x == 0) {
        f.part[g.N + blockIdx.y] = any_bad ? 1.0 : 0.0;
        __threadfence();
        s_last = (atomicAdd(&f.tickets[0], 1u) == (unsigned)(n_cta - 1));
    }
    __syncthreads();
    if (!s_last) return;
    __threadfence();
    // the per-sample sums and the per-CTA flags come back through the warp (independent loads), then thread 0 adds in sample order
    __shared__ double s_part[kMaxSamples];
    for (int t = threadIdx.x; t < g.N; t += blockDim.x) s_part[t] = __ldcg(&f.part[t]);
    int bad_l = 0;
    for (int cta = threadIdx.x; cta < n_cta; cta += blockDim.x) bad_l |= __ldcg(&f.part[g.N + cta]) != 0.0;
    const bool bad = __syncthreads_or(bad_l) != 0;
    if (threadIdx.x == 0) {
        f.tickets[0] = 0u;                               // re-arm for the next launch
        if (fcommit) {
            if (phase_in == 1) {                         // the incoming iterate closes an outer iteration
                state_close_outer(st, f, cf_new, a.tol);
                if (fstop) return;                       // the same test as state_close_outer's, taken by every CTA above
            }
            st->u_cur = ucur_in ^ 2;                     // commit the U step of the fused pass
            state_end_u(st, a.mom_a[tu_in + n2], tu_in + n2, lw_pass, n2 > 0);
            st->phase = 1;
        }
        if (bad) st->done = 3;
        if (sharded) state_u_norm(st, f.rscal[4]);
        double sa = 0.0;
        for (int t = 0; t < g.N; ++t) sa += s_part[t];
        state_end_alpha(st, sa, !fw, a.mom_a[t0 + n2], t0 + n2, l_h, n2 > 0);
    }
}

#ifndef DMF_INST_BODY     // launched by dmf_api.cu only: the instantiation units leave these kernels out
// ------------------------------------------------------------------------------------------------
// CpG rows sharded over GPUs: the set-up / termination logic of the rowgram pass on the all-reduced sums
// FitDev::rscal = [cost, ||R_trunc||^2, ||u||^2, max d_x] (deconvolution.py:192-204, :218-221).  One thread per fit.
static __global__ void finalize_cost_kernel(const PassArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.k_inner) return;
    const FitDev f = a.fits[i];
    FitState* st = f.st;
    if (st->done) return;
    if (a.flags & kFlagInitial) {
        const size_t slot = (size_t)st->a_cur * a.g.Kt * a.g.N;
        if (a.flags & kFlagF32) state_setup(st, f, f.rscal, f.rscal[3], a.g, reinterpret_cast<const float*>(f.A) + slot);
        else state_setup(st, f, f.rscal, f.rscal[3], a.g, reinterpret_cast<const double*>(f.A) + slot);
    } else {
        state_close_outer(st, f, f.rscal[0], a.tol);
    }
}

// CpG rows sharded over GPUs, stream engine: the end of a U step on the all-reduced ||u||^2 (FitDev::rscal[4]).  One thread per fit.
static __global__ void u_commit_kernel(const PassArgs a) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.k_inner) return;
    const FitDev f = a.fits[i];
    if (f.st->done) return;
    state_u_norm(f.st, f.rscal[4]);
}

// CpG rows sharded over GPUs, stream engine: the step of alpha_pass_kernel on the all-reduced gradient (the first Kt*N doubles of
// FitDev::rgram).  One CTA per fit.
static __global__ void __launch_bounds__(kThreads) alpha_commit_kernel(const PassArgs a) {
    __shared__ double colred[kMaxSamples];
    const FitDev f = a.fits[blockIdx.x];
    if (f.st->done) return;
    const bool fw = (a.flags & kFlagFW) != 0;
    if (a.flags & kFlagF32) alpha_step<float>(a.g, f, f.rgram, colred, fw, a.k_inner);
    else alpha_step<double>(a.g, f, f.rgram, colred, fw, a.k_inner);
}

// ------------------------------------------------------------------------------------------------
// CpG rows sharded over GPUs: all-reduce of the statistics block over NVLink PEER MEMORY, in one kernel and without NCCL.
// Every rank owns a symmetric buffer  data[2 parities][world slots][n] + flags[2][world]  that all ranks of the box can address
// (torch symmetric memory / cuMem peer mappings).  One launch per rank:
//   1. push   : the rank's local sums go into slot [rank] of EVERY rank's buffer (plain st.global over NVLink, 16-byte vectors)
//   2. signal : after a system-scope fence the last CTA stores the epoch into flag [rank] of every rank
//   3. wait   : every CTA spins (ld.acquire.sys) until all `world` flags of ITS OWN buffer show the epoch
//   4. sum    : slots are added in rank order (the same order on every rank -> bit-identical results everywhere) into the
//               `global` statistics block that alpha_inner_kernel / finalize_cost_kernel read
// Two parities alternate with the epoch: a rank can only be one exchange ahead of a peer (it needs the peer's flag of epoch e
// before it can push e + 1), so a slot is never overwritten while its owner still sums it.
struct XchgArgs {
    double* const* peers;     // device array [world]: base of rank r's symmetric buffer as mapped in this process
    const double* local;      // this rank's statistics blocks (n_fits x per_fit doubles)
    double* global;           // all-reduced copies, same layout
    unsigned* ticket;         // grid-completion ticket (zeroed at set-up, re-armed by the last CTA)
    long long per_fit;        // doubles per fit in local / global
    long long slot_stride;    // doubles per slot of the symmetric buffer (>= n_fits * per_fit)
    long long flag_off;       // byte offset of the flags inside a symmetric buffer
    long long scal_off;       // offset of the 8 scalars inside a fit's block
    int n_fits, rank, world;
    int which;                // 0: whole blocks; 1: the 8 scalars of every fit (sum); 2: the same at set-up (slot 3 = max d_x: max)
    unsigned* epoch_dev;      // exchanges completed so far (device memory, so that a captured launch advances with every replay);
                              // ticket[1] counts the CTAs that finished the exchange
};

__device__ __forceinline__ void st_release_sys(unsigned* p, unsigned v) { asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory"); }
__device__ __forceinline__ unsigned ld_acquire_sys(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

static __global__ void __launch_bounds__(kThreads) peer_allreduce_kernel(const XchgArgs a) {
    __shared__ int s_last;
    const unsigned epoch = *reinterpret_cast<volatile unsigned*>(a.epoch_dev) + 1u;     // the last CTA to leave publishes it (below)
    const int parity = epoch & 1u;
    const long long n = a.which == 0 ? (long long)a.n_fits * a.per_fit : (long long)a.n_fits * 8;
    const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nthr = (long long)gridDim.x * blockDim.x;
    auto src_index = [&](long long e) { return a.which == 0 ? e : (e >> 3) * a.per_fit + a.scal_off + (e & 7); };
    // 1. push my sums into slot [rank] of every rank's buffer
    for (int p = 0; p < a.world; ++p) {
        double* dst = a.peers[(p + a.rank) % a.world] + ((long long)parity * a.world + a.rank) * a.slot_stride;     // staggered peer order
        for (long long e = tid; e < n; e += nthr) dst[e] = a.local[src_index(e)];
    }
    // 2. signal
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) s_last = (atomicAdd(a.ticket, 1u) == gridDim.x - 1);
    __syncthreads();
    if (s_last) {
        __threadfence_system();
        if (threadIdx.x < a.world) {
            unsigned* flags = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(a.peers[threadIdx.x]) + a.flag_off);
            st_release_sys(flags + parity * a.world + a.rank, epoch);
        }
        if (threadIdx.x == 0) *a.ticket = 0u;
    }
    // 3. wait for every rank's flag in MY buffer
    if (threadIdx.x < a.world) {
        const unsigned* flags = reinterpret_cast<const unsigned*>(reinterpret_cast<const char*>(a.peers[a.rank]) + a.flag_off);
        while (ld_acquire_sys(flags + parity * a.world + threadIdx.x) != epoch) { __nanosleep(64); }
    }
    __syncthreads();
    // 4. rank-ordered sum (L1 bypassed: the slots were written by peers)
    const double* mine = a.peers[a.rank] + (long long)parity * a.world * a.slot_stride;
    for (long long e = tid; e < n; e += nthr) {
        double s = __ldcg(mine + e);
        const bool is_max = a.which == 2 && (e & 7) == 3;
        for (int r = 1; r < a.world; ++r) {
            const double v = __ldcg(mine + (long long)r * a.slot_stride + e);
            s = is_max ? fmax(s, v) : s + v;
        }
        a.global[src_index(e)] = s;
    }
    // every CTA read the count at entry; the last one to get here advances it for the next launch (stream order separates launches)
    __syncthreads();
    if (threadIdx.x == 0 && atomicAdd(a.ticket + 1, 1u) == gridDim.x - 1) {
        a.ticket[1] = 0u;
        *a.epoch_dev = epoch;
    }
}
#endif  // DMF_INST_BODY

}  // namespace dmf
