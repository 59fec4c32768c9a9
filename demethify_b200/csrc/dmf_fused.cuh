// dmf_fused.cuh — "fused" engine: ONE streaming pass over X, d_x, R_trunc, u per OUTER iteration of
// deconvolution.py:206-221 (SURVEY.md 7.1 #1-#3, 8 d4 "fused outer iteration").
//
// The Gram-form engine (dmf_gram.cuh) needs two passes per outer iteration because the panel statistics of the alpha step
// need the u that the U step produces.  The U step is row-local, so a row tile can go through all three stages on one visit:
//
//   A  row statistics   c = x - R_trunc a_k,  b_m = (d o c) a_u^T,  H_m = a_u diag(d_m) a_u^T   (+ sum d c^2 for the cost)
//   U  n_iter2 update_u iterations per row on (b_m, H_m)  (deconvolution.py:82-89 / :157-164), the row's cost cross terms
//      -2 u^T b_m + u^T H_m u of the INCOMING iterate, the new (u, u_) written to the other slot pair
//   C  Gram panel with the NEW u:  G_uk += d (u (x) R_trunc),  G_uu += d (u (x) u),  bx_u += (d o x) u
//
// The cost of the incoming iterate (u_k, alpha_k) is complete at the end of the pass; the last CTA then runs the termination
// test of deconvolution.py:218-221 for outer iteration k and COMMITS the U step (flips the slot pair, publishes the panel,
// updates l_h, a1) only if the fit did not just terminate - so a terminated fit returns exactly the iterate whose cost passed
// the test.  alpha_inner_kernel (dmf_gram.cuh) follows and produces alpha_{k+1}.
//
// One CTA = 20 (or 24) warps with four roles (warp specialised, tiles flow A -> U -> C through a shared-memory ring; rows per tile,
// ring depth, warp maps and the number of U-warps depend on the width class - FusedCfg below):
//   8 A-warps   row blocks x sample groups; c comes from FP64 tensor-core MMAs (mma.sync.m8n8k4.f64, SASS DMMA) with the ROWS on
//               the M side: a lane owns one row and two samples of every 8-sample block; the row statistics run on the FMA pipe
//   3 (7) U-warps  lane = row (one unknown type) or (row, component) (two); work unit n goes to U-warp n mod FU (the 20 dependent
//               iterations of a unit take longer than the A and C stages of a tile, so consecutive tiles must overlap)
//   1 producer  drives the TMA ring: one bulk copy per matrix and tile into bank-conflict-free padded rows
//   8 C-warps   the panel is the GEMM  [N x rows] (d) x [rows x NCOL] (u (x) [R_trunc | u]) : DMMA again, accumulators stay in
//               the MMA C fragments for the whole kernel; bx_u on the FMA pipe
// FP64 only (tcgen05 has no FP64 kind; DMMA and DFMA share one pipe at 64 FMA/clk/SM - tools/fp64_peak.cu), which is the
// binding roofline of this kernel: ~39 FMA per (row, sample) against 10 bytes.
#pragma once
#include <type_traits>
#include "dmf_gram.cuh"

namespace dmf {

#ifndef DMF_FU
#define DMF_FU 3
#endif
#ifndef DMF_FU_NARROW
#define DMF_FU_NARROW 3
#endif
#ifndef DMF_FU_NARROW2
#define DMF_FU_NARROW2 7
#endif
#ifndef DMF_STAGES
#define DMF_STAGES 5
#endif
constexpr int kFA = 8, kFC = 8, kFP = 1;
// Registers per thread after the role split (setmaxnreg).  The pool is what the CTA got at launch (threads x the register count ptxas
// derives from __launch_bounds__): 20 warps -> 96 per thread, 24 warps -> 80 per thread.  With 3 U-warps: A 88, C 96 (measured at 1M x 256: A 88 0.788 ms, 96 0.797, 104 0.831, 112 0.824, 80 0.871; C 112 spills more and is no faster), U / producer 64
// (256 (88 + 96) + 128 x 64 <= 640 x 96); with 7 U-warps: A 88, C 96, U / producer 56 (256 (88 + 96) + 256 x 56 = 768 x 80).
// setmaxnreg is a warpgroup instruction: the warp count must stay a multiple of 4 (FU = 3 or 7) so that every group is one role set.
#ifndef DMF_RA
#define DMF_RA 88
#endif
#ifndef DMF_RC
#define DMF_RC 96
#endif
constexpr int kFusedMaxU = 7;
constexpr int fused_launch_regs(int threads) { return (65536 / ((threads + 127) / 128 * 128)) / 8 * 8; }
template <int FROM, int TO>
__device__ __forceinline__ void fused_set_regs() {
    if constexpr (TO > FROM) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(TO));
    else if constexpr (TO < FROM) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(TO));
}
// Tile geometry by the width class S (N <= 64 S samples).  The 20 dependent update_u iterations of a tile take the same time
// whatever N is, while the A / C work of a row shrinks with N: narrow problems get 32-row tiles (a U-warp pass uses all 32 lanes
// when there is one unknown type, two U-warps share a tile when there are two), one more U-warp and - their stages being small -
// a deeper ring, so that enough tiles are in flight to cover the U latency.
//   S = 4: 16-row tiles, A-warps = 2 row blocks x 4 sample groups (8 blocks of 8 samples each), C-warps = 8 sample groups x 4 k-steps
//   S = 2: 32-row tiles, A-warps = 4 row blocks x 2 sample groups (8 blocks),                   C-warps = 4 sample groups x 2 row splits x 4 k-steps
//   S = 1: 32-row tiles, A-warps = 4 row blocks x 2 sample groups (4 blocks),                   C-warps = 2 sample groups x 4 row splits x 2 k-steps
template <int S, int NUB>
struct FusedCfg {
    static constexpr int TR = S == 4 ? 16 : 32;                        // rows per tile
    // U-warps: a pass of two unknown types covers 16 rows only, so narrow problems with n_u = 2 get 7 U-warps (measured: 500k x 64,
    // n_u = 2: 0.201 -> 0.171 ms; 500k x 128: 0.265 -> 0.246 ms; no gain for one unknown type)
    static constexpr int FU = S == 4 ? DMF_FU : (NUB == 2 ? DMF_FU_NARROW2 : DMF_FU_NARROW);
    static constexpr int NS = S == 4 ? DMF_STAGES : (S == 2 ? 4 : 8);  // ring stages
    static constexpr int RB = TR / 8, SG = 8 / RB, NSB = 8 * S / SG;   // A-warps: row blocks x sample groups, 8-sample blocks per warp
    static constexpr int CSG = 2 * S, RSP = 8 / CSG, KSW = (TR / 4) / RSP;   // C-warps: 32-sample groups x row splits, k-steps (4 rows) per warp
    static constexpr int WARPS = kFA + kFC + FU + kFP, THREADS = WARPS * 32;
    static constexpr int LR = fused_launch_regs(THREADS);              // registers per thread at launch
    static constexpr int RA = FU >= 5 ? 88 : DMF_RA, RC = FU >= 5 ? 96 : DMF_RC, RU = FU >= 5 ? 56 : 64;
    static_assert(FU <= kFusedMaxU && WARPS % 4 == 0 && RA % 8 == 0 && RC % 8 == 0 && 256 * (RA + RC) + 32 * (FU + 1) * RU <= THREADS * LR,
                  "register split of the fused pass");
    // row-statistics buffers: S = 4 double-buffers them (released through `sfree` as soon as the U-warp holds the partials in
    // registers: shared memory is full there); the narrow classes keep one per stage (released with the stage)
    static constexpr int NSTAT = S == 4 ? 2 : NS;
    static constexpr int UP = NUB == 2 ? TR / 16 : 1;                  // U work units per tile (16 rows x 2 components, or all rows)
    // The mbarrier waits are by phase PARITY: a U-warp that moves from tile t to tile t + ceil(FU / UP) must not find the stage of the
    // new tile two fills behind, or the parity test passes on the wrong fill (stale statistics, then a deadlock - seen with
    // FU = 7 at S = 4).  Fills are in tile order, so a stride of at most NS tiles guarantees it.
    static_assert((FU + UP - 1) / UP <= NS, "U-warp tile stride must not exceed the ring depth (parity waits)");
};
// The host's view of FusedCfg for the instantiated classes (S = 1, 2, 4; one or two unknown types)
struct FusedShape { int rows, stages, threads, sgroups, nstat; };
template <int S, int NUB>
constexpr FusedShape fused_shape_of() { using C = FusedCfg<S, NUB>; return {C::TR, C::NS, C::THREADS, C::SG, C::NSTAT}; }
inline FusedShape fused_shape(int s, int nub) {
    switch (s * 10 + nub) {
        case 11: return fused_shape_of<1, 1>();
        case 12: return fused_shape_of<1, 2>();
        case 21: return fused_shape_of<2, 1>();
        case 22: return fused_shape_of<2, 2>();
        case 41: return fused_shape_of<4, 1>();
        case 42: return fused_shape_of<4, 2>();
    }
    return FusedShape{};
}
constexpr int kFusedMaxInner = 64;       // beyond this the U-warps would bound the pass: Gram engine instead
constexpr unsigned kFusedCtlBytes = 2048;

struct FusedArgs {
    Geom g;                  // problem sizes, pitches, n_parts / n_groups / part_stride of this launch
    const FitDev* fits;
    int n_iter2, flags;
    double tol;
    const double* mom_a;
    const double* mom_m;
    int n_tiles;
    unsigned pitchX, pitchD;                          // bytes per row of X / d_x, in global and in shared memory
    unsigned offD, offR, offU, offUp, stage_bytes;    // stage layout, X at 0
    unsigned offStats, offTab;                        // from the start of dynamic shared memory
    unsigned zero_off;                                // offset (inside a stage) of 8 bytes that always hold 0.0
};
typedef void (*fused_kern_t)(const FusedArgs);

struct FusedCtl {
    unsigned long long full[8], empty[8], stats[8], udone[8], sfree[2];
    double wsum[2][kFA + kFC + kFusedMaxU + kFP];
    double beta[2 * kFusedMaxInner];      // (1 + beta_t, -beta_t) of this launch's update_u iterations (the same for every row)
    int flag, commit;
};
static_assert(sizeof(FusedCtl) <= kFusedCtlBytes, "fused control block too large");

// D (8 x 8) += A (8 x 4, lane holds A[lane / 4][lane % 4]) x B (4 x 8, lane holds B[lane % 4][lane / 4]); the lane's two
// accumulators are D[lane / 4][2 (lane % 4)] and D[lane / 4][2 (lane % 4) + 1]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
    asm("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// two adjacent weights (same row, samples j and j + 1; j even) as doubles
template <typename WT>
__device__ __forceinline__ void lds_weight2(uint32_t addr, double& d0, double& d1);
template <>
__device__ __forceinline__ void lds_weight2<uint16_t>(uint32_t addr, double& d0, double& d1) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    d0 = (double)(v & 0xffffu);
    d1 = (double)(v >> 16);
}
template <>
__device__ __forceinline__ void lds_weight2<double>(uint32_t addr, double& d0, double& d1) { lds2(addr, d0, d1); }

// np.clip(., 0, 1) by two comparisons of the SAME value (they issue together; a NaN fails both and propagates, as in numpy;
// the simplex projection of the alpha step then stops the fit)
__device__ __forceinline__ double clip01_keepnan(double v) {
    double r = v > 1.0 ? 1.0 : v;
    return v < 0.0 ? 0.0 : r;
}
// The same clip on the integer pipe, for FINITE v (the U-warps check once per tile that every iterate stays finite): every
// FP64 instruction of a U-warp queues behind the DMMAs of the other 16 warps, integer compares do not.
//   v < 0  <=>  sign bit set (-0.0 -> 0.0, equal);   v > 1  <=>  sign clear and bits > bits(1.0)
__device__ __forceinline__ double clip01_finite(double v) {
    const long long b = __double_as_longlong(v);
    const bool big = (unsigned long long)b > 0x3FF0000000000000ull;
    const bool neg = b < 0;
    const long long r = neg ? 0ll : (big ? 0x3FF0000000000000ll : b);
    return __longlong_as_double(r);
}

// One update_u step of deconvolution.py:82-89 (gradient at u for the unsupervised variant, :163) on the row's statistics,
// (prev, cur) -> next.  The U-warps run 16 rows x n_iter2 of these back to back while the other 16 warps of the CTA keep the
// FP64 pipe busy - every FP64 instruction queues behind their DMMAs - so both the DEPTH of the chain from cur to next and the
// NUMBER of FP64 instructions count.  With  Mh = H / l_w,  c = b / l_w  and  Am = I - Mh  (per row, once):
//     u_t = u + beta (u - u_)                        ->  fma(1 + beta, u, (-beta) u_)      ((-beta) u_ does not depend on u)
//     u_t + (b - H u_t) / l_w  =  Am u_t + c         ->  fma(Am_qq, u_t[q], fma(Am_qq', u_t[q'], c_q))
// i.e. 3 dependent FP64 operations per iteration instead of 9 and the clip on the integer pipe; the roundings differ from the
// reference's operation order by ~1 ulp of u per iteration, the same size as the reference's own rounding of u_t + step.
// bt = (1 + beta_t, -beta_t) from shared memory.
template <bool AT_CURRENT, bool FINITE, int NUB>
__device__ __forceinline__ void fused_u_step(const double (&pv)[NUB], const double (&cu)[NUB], const double (&am)[NUB][NUB],
                                             const double (&c)[NUB], double opb, double nbeta, double (&nx)[NUB]) {
    double ut[NUB];
#pragma unroll
    for (int q = 0; q < NUB; ++q) ut[q] = fma(opb, cu[q], nbeta * pv[q]);
#pragma unroll
    for (int q = 0; q < NUB; ++q) {
        double un;
        if (AT_CURRENT) {        // gradient at u (deconvolution.py:163): am = -Mh
            double gq = c[q];
#pragma unroll
            for (int q2 = 0; q2 < NUB; ++q2) gq = fma(am[q][q2], cu[q2], gq);
            un = ut[q] + gq;
        } else {                 // am = I - Mh
            un = c[q];
#pragma unroll
            for (int q2 = 0; q2 < NUB; ++q2)
                if (q2 != q) un = fma(am[q][q2], ut[q2], un);
            un = fma(am[q][q], ut[q], un);
        }
        nx[q] = FINITE ? clip01_finite(un) : clip01_keepnan(un);
    }
}
// n2 steps, two at a time so that (u_, u) rotate without register copies; (1 + beta_t, -beta_t) come from shared memory
template <bool AT_CURRENT, bool FINITE, int NUB>
__device__ __forceinline__ void fused_u_loop(double (&u)[NUB], double (&up)[NUB], const double (&am)[NUB][NUB], const double (&c)[NUB],
                                             uint32_t beta32, int n2) {
    int itn = 0;
    for (; itn + 2 <= n2; itn += 2) {
        double o0, b0, o1, b1, n1[NUB], n3[NUB];
        lds2(beta32 + (uint32_t)itn * 16u, o0, b0);
        lds2(beta32 + (uint32_t)itn * 16u + 16u, o1, b1);
        fused_u_step<AT_CURRENT, FINITE, NUB>(up, u, am, c, o0, b0, n1);
        fused_u_step<AT_CURRENT, FINITE, NUB>(u, n1, am, c, o1, b1, n3);
#pragma unroll
        for (int q = 0; q < NUB; ++q) { up[q] = n1[q]; u[q] = n3[q]; }
    }
    if (itn < n2) {
        double o0, b0, n1[NUB];
        lds2(beta32 + (uint32_t)itn * 16u, o0, b0);
        fused_u_step<AT_CURRENT, FINITE, NUB>(up, u, am, c, o0, b0, n1);
#pragma unroll
        for (int q = 0; q < NUB; ++q) { up[q] = u[q]; u[q] = n1[q]; }
    }
}
template <bool AT_CURRENT, int NUB>
__device__ __forceinline__ void fused_u_iterate(double (&u)[NUB], double (&up)[NUB], const double (&v)[ng_of(NUB)], uint32_t beta32, int n2,
                                                double inv_lw) {
    double am[NUB][NUB], c[NUB];
    // every iterate stays finite (|u_next| <= |Am| |u_t| + |c| with |u_t| <= 3) when the row's constants and the incoming pair are
    // moderate: then the clip runs on the integer pipe; otherwise (l_w = 0, NaN / Inf in the data) the comparisons keep numpy's NaN rules
    bool tame = true;
#pragma unroll
    for (int q = 0; q < NUB; ++q) {
        c[q] = v[q] * inv_lw;
        tame = tame && fabs(c[q]) < 1e150 && fabs(u[q]) <= 1.0 && fabs(up[q]) <= 1.0;
#pragma unroll
        for (int q2 = 0; q2 < NUB; ++q2) {
            const double mh = v[NUB + (q <= q2 ? tri_index(q, q2, NUB) : tri_index(q2, q, NUB))] * inv_lw;
            am[q][q2] = (!AT_CURRENT && q == q2) ? 1.0 - mh : -mh;
            tame = tame && fabs(mh) < 1e150;
        }
    }
    if (__all_sync(0xffffffffu, tame)) fused_u_loop<AT_CURRENT, true, NUB>(u, up, am, c, beta32, n2);
    else fused_u_loop<AT_CURRENT, false, NUB>(u, up, am, c, beta32, n2);
}

// Two unknown types: the two components of a row live in lanes (row, row + 16), so a U-warp issues half as many FP64 instructions
// per iteration (each of them queues behind the DMMAs of the other warps) and uses all 32 lanes; the other component's u_t
// (u at :163) comes through one shuffle.  cu / pv: own component of (u, u_); on return (u_new, previous u_new).
template <bool AT_CURRENT, bool FINITE>
__device__ __forceinline__ void fused_u_loop_split(double& cu, double& pv, double am_own, double am_oth, double c, uint32_t beta32, int n2) {
    for (int itn = 0; itn < n2; ++itn) {
        double opb, nbeta, un;
        lds2(beta32 + (uint32_t)itn * 16u, opb, nbeta);
        const double ut = fma(opb, cu, nbeta * pv);
        if (AT_CURRENT) {
            const double cuo = __shfl_xor_sync(0xffffffffu, cu, 16);
            un = ut + fma(am_oth, cuo, fma(am_own, cu, c));
        } else {
            const double t = fma(am_own, ut, c);
            const double uto = __shfl_xor_sync(0xffffffffu, ut, 16);
            un = fma(am_oth, uto, t);
        }
        pv = cu;
        cu = FINITE ? clip01_finite(un) : clip01_keepnan(un);
    }
}

// A-warps: row statistics of ONE row (the lane's, rows on the M side of the MMA) over the warp's NSB blocks of 8 samples; the lane
// owns samples 2 ti, 2 ti + 1 of every block.  xa / da: the lane's row at the warp's first block, sample 2 ti; ta: the lane's pair
// record [a_u(j) | a_u(j + 1)] of the per-sample table.  The shared-memory data pipe is the busiest unit of this kernel after the
// FP64 pipe, so the table holds a_u only and the H terms go through w_q = d a_u[q]:  b_q += w_q c,  H_qq' += w_q a_u[q'].
// MASK: the tile is short or some of the warp's samples do not exist (nblk = existing blocks, jlane = first block's sample 2 ti).
// acc = [b (NUB) | H upper triangle] of the row.
template <bool MASK, typename WT, int KS, int NUB, int NSB>
__device__ __forceinline__ void fused_row_stats(uint32_t xa, uint32_t da, uint32_t ta, const double (&rfrag)[KS > 0 ? KS : 1],
                                                const double (&nab)[NSB][KS > 0 ? KS : 1], int nblk, int jlane, int N, bool live,
                                                double& cost, double (&acc)[ng_of(NUB)]) {
#pragma unroll
    for (int sb = 0; sb < NSB; ++sb) {
        if (MASK && sb >= nblk) break;
        double c0, c1, d0, d1, au0[NUB], au1[NUB];
        lds2(xa + (uint32_t)sb * 64u, c0, c1);
        lds_weight2<WT>(da + (uint32_t)sb * 8u * (unsigned)sizeof(WT), d0, d1);
        if (NUB == 1) lds2(ta + (uint32_t)sb * 64u, au0[0], au1[0]);
        else {
#pragma unroll
            for (int i = 0; i < NUB / 2; ++i) {
                lds2(ta + (uint32_t)sb * (4u * 2u * NUB * 8u) + (uint32_t)i * 16u, au0[2 * i], au0[2 * i + 1]);
                lds2(ta + (uint32_t)sb * (4u * 2u * NUB * 8u) + (uint32_t)(NUB / 2 + i) * 16u, au1[2 * i], au1[2 * i + 1]);
            }
        }
        if (MASK) {
            const bool v0 = jlane + 8 * sb < N, v1 = jlane + 8 * sb + 1 < N;
            if (!v0) c0 = 0.0;
            if (!v1) c1 = 0.0;
            if (!(v0 && live)) d0 = 0.0;
            if (!(v1 && live)) d1 = 0.0;
        }
        // c = x - R_trunc a_k.  With two k-steps the second accumulates on its own and one DADD per value joins them: a dependent
        // DMMA pair would hold the warp for the full MMA latency (measured with C at 96 registers: 0.847 -> 0.837 ms at 1M x 256)
        if (KS == 2) {
            double e0 = 0.0, e1 = 0.0;
            dmma884(c0, c1, rfrag[0], nab[sb][0]);
            dmma884(e0, e1, rfrag[KS - 1], nab[sb][KS - 1]);
            c0 += e0;
            c1 += e1;
        } else {
#pragma unroll
            for (int kk = 0; kk < KS; ++kk) dmma884(c0, c1, rfrag[kk], nab[sb][kk]);
        }
        const double z0 = d0 * c0, z1 = d1 * c1;
        cost = fma(z0, c0, cost);
        cost = fma(z1, c1, cost);
#pragma unroll
        for (int q = 0; q < NUB; ++q) {
            const double w0 = d0 * au0[q], w1 = d1 * au1[q];
            acc[q] = fma(w0, c0, acc[q]);
            acc[q] = fma(w1, c1, acc[q]);
#pragma unroll
            for (int q2 = q; q2 < NUB; ++q2) {
                acc[NUB + tri_index(q, q2, NUB)] = fma(w0, au0[q2], acc[NUB + tri_index(q, q2, NUB)]);
                acc[NUB + tri_index(q, q2, NUB)] = fma(w1, au1[q2], acc[NUB + tri_index(q, q2, NUB)]);
            }
        }
    }
}

// C-warps: KSW k-steps (4 rows each) of one tile of the Gram panel with the new u, for the warp's 32 samples.  The lane's samples
// are jb + 16 h + 2 gi + e (mb = 2 h + e is the MMA block, gi the row of the A fragment), so x and d come as pairs; k-step ks
// covers tile rows 8 (ks / 2) + (ks % 2) + 2 ti (bank-conflict free with the recommended pitches).  The B operand is
// u_q (x) W with W = [R_trunc | u] (KB + NUB columns, WB blocks of 8): block nb = q WB + wb, column gi = u_q W[8 wb + gi]; the lane
// reads its W entry from the stage (w_off / w_pitch; columns that do not exist point at a zero with pitch 0).
template <bool MASK, typename WT, int NUB, int KSW, int WB>
__device__ __forceinline__ void fused_panel_tile(const FusedArgs& a, uint32_t sb32, int nrows, int ti, int ks0, uint32_t xoff, uint32_t doff,
                                                 const unsigned (&w_off)[WB], const unsigned (&w_pitch)[WB], const bool (&valid)[4],
                                                 double (&acc)[4][NUB * WB][2], double (&accx)[4][NUB]) {
    const unsigned upitch = (unsigned)(a.g.ldu * 8);
#pragma unroll
    for (int i = 0; i < KSW; ++i) {
        const int ks = ks0 + i;
        const int row = 8 * (ks >> 1) + (ks & 1) + 2 * ti;
        const bool lrow = row < nrows;
        double bfrag[NUB * WB], un[NUB], w[WB];
        if (NUB == 2) lds2(sb32 + a.offU + (uint32_t)row * upitch, un[0], un[NUB - 1]);
        else {
#pragma unroll
            for (int q = 0; q < NUB; ++q) lds1(sb32 + a.offU + (uint32_t)row * upitch + (uint32_t)q * 8u, un[q]);
        }
#pragma unroll
        for (int wb = 0; wb < WB; ++wb) lds1(sb32 + w_off[wb] + (uint32_t)row * w_pitch[wb], w[wb]);
#pragma unroll
        for (int q = 0; q < NUB; ++q)
#pragma unroll
            for (int wb = 0; wb < WB; ++wb) bfrag[q * WB + wb] = un[q] * w[wb];
        const uint32_t xr = sb32 + (uint32_t)row * a.pitchX + xoff;
        const uint32_t dr = sb32 + a.offD + (uint32_t)row * a.pitchD + doff;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            double x0, x1, d0, d1;
            lds2(xr + (uint32_t)h * 128u, x0, x1);
            lds_weight2<WT>(dr + (uint32_t)h * 16u * (unsigned)sizeof(WT), d0, d1);
            if (MASK) {
                if (!(valid[2 * h] && lrow)) { d0 = 0.0; x0 = 0.0; }
                if (!(valid[2 * h + 1] && lrow)) { d1 = 0.0; x1 = 0.0; }
            }
            const double dx0 = d0 * x0, dx1 = d1 * x1;
#pragma unroll
            for (int q = 0; q < NUB; ++q) {
                accx[2 * h][q] = fma(dx0, un[q], accx[2 * h][q]);
                accx[2 * h + 1][q] = fma(dx1, un[q], accx[2 * h + 1][q]);
            }
#pragma unroll
            for (int nb = 0; nb < NUB * WB; ++nb) {
                dmma884(acc[2 * h][nb][0], acc[2 * h][nb][1], d0, bfrag[nb]);
                dmma884(acc[2 * h + 1][nb][0], acc[2 * h + 1][nb][1], d1, bfrag[nb]);
            }
        }
    }
}

template <typename WT, int KB, int NUB, int S>
__global__ void __launch_bounds__((FusedCfg<S, NUB>::THREADS), 1) fused_outer_kernel(const FusedArgs a) {
    extern __shared__ __align__(128) unsigned char smem[];
    using Cfg = FusedCfg<S, NUB>;
    constexpr int KS = (KB + 3) / 4;                  // k-steps of the c = x - R_trunc a_k MMA
    constexpr int NG = ng_of(NUB);
    constexpr int NTRI = NG - NUB;
    constexpr int NCOL = NUB * KB + NTRI;             // panel columns: u_q R_k (q major), then the upper triangle of u u^T
    constexpr int WB = (KB + NUB + 7) / 8;            // blocks of 8 columns of W = [R_trunc | u]; the panel MMA runs u_q (x) W per q
    constexpr int NBLK = NUB * WB;
    constexpr int NS = Cfg::NS, TR = Cfg::TR, FU = Cfg::FU, THREADS = Cfg::THREADS;
    constexpr int NSB = Cfg::NSB;                     // A-warp: 8 rows x NSB blocks of 8 samples
    constexpr int SG = Cfg::SG;                       // partial statistics records per row (one per A-warp sample group)
    constexpr int RSP = Cfg::RSP, KSW = Cfg::KSW;     // C-warp: 32 samples x KSW k-steps (CSG sample groups x RSP row splits)
    constexpr int UP = Cfg::UP;                       // U work units per tile
    constexpr unsigned STATB = (unsigned)(SG * TR * NG) * 8u;   // bytes of one row-statistics buffer
    constexpr unsigned PAIRB = 2u * NUB * 8u;         // bytes of one pair record of the per-sample table
    const Geom& g = a.g;
    const FitDev f = a.fits[fit_id(g)];
    FitState* st = f.st;
    if (st->done) return;
    FusedCtl* ctl = reinterpret_cast<FusedCtl*>(smem);
    const int tid = threadIdx.x, lane = tid & 31;
    const int warp = tid >> 5;
    const int gi = lane >> 2, ti = lane & 3;
    const uint32_t smem32 = smem_u32(smem);
    const uint32_t stages32 = smem32 + kFusedCtlBytes;
    const int part = part_id(g);
    const int n_my = (a.n_tiles > part) ? (a.n_tiles - part + g.n_parts - 1) / g.n_parts : 0;
    const int ucur = st->u_cur, acur = st->a_cur;
    const double* Acur = reinterpret_cast<const double*>(f.A) + (size_t)acur * g.Kt * g.N;
    const int N = g.N, K = g.K;

    if (tid == 0) {
#pragma unroll
        for (int s = 0; s < NS; ++s) {
            mbar_init(smem_u32(&ctl->full[s]), 1);
            mbar_init(smem_u32(&ctl->empty[s]), kFC);
            mbar_init(smem_u32(&ctl->stats[s]), kFA * 8);      // the 8 writer lanes of every A-warp
            mbar_init(smem_u32(&ctl->udone[s]), UP);
        }
        mbar_init(smem_u32(&ctl->sfree[0]), 1);
        mbar_init(smem_u32(&ctl->sfree[1]), 1);
        mbar_fence_init();
    }
    // every stage starts as finite data: rows beyond the end of the last tile and samples beyond N are weighted with d = 0,
    // which only works on finite values
    {
        const unsigned n16 = (a.offStats - kFusedCtlBytes) / 16;
        for (unsigned i = tid; i < n16; i += THREADS)
            asm volatile("st.shared.v4.u32 [%0], {%1, %1, %1, %1};" ::"r"(stages32 + i * 16u), "r"(0u) : "memory");
    }
    // per-sample table of the A-warps, one record per pair of samples: [a_u(j) | a_u(j + 1)], zero beyond N
    for (int p = tid; p < 32 * S; p += THREADS) {
        double* rec = reinterpret_cast<double*>(smem + a.offTab + (size_t)p * PAIRB);
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int j = 2 * p + e;
#pragma unroll
            for (int q = 0; q < NUB; ++q) rec[e * NUB + q] = (j < N && q < g.nu) ? Acur[(size_t)(K + q) * N + j] : 0.0;
        }
    }
    if (tid < a.n_iter2) {
        // beta_t = min((a_t - 1) / a_{t+1}, 0.9999 sqrt(l_w_ / l_w)); l_w_ == l_w from the second inner iteration on (:89)
        const double l_w = st->l_w;
        const double cap = 0.9999 * sqrt((tid == 0 ? st->l_w_old : l_w) / l_w);
        const double bt = fmin(a.mom_m[st->t_u + tid], cap);
        ctl->beta[2 * tid] = 1.0 + bt;
        ctl->beta[2 * tid + 1] = -bt;
    }
    fence_proxy_async_smem();
    __syncthreads();

    // only the last tile of the matrix can be short; it is local tile it_short of the CTA that owns it
    const int rows_last = (int)(g.M - (long long)(a.n_tiles - 1) * TR);
    const int it_short = (rows_last < TR && (a.n_tiles - 1) % g.n_parts == part) ? (a.n_tiles - 1) / g.n_parts : -1;
    auto tile_rows = [&](int it) { return it == it_short ? rows_last : TR; };

    double cost = 0.0, ssq = 0.0;       // per-thread partials (A-warps: sum d c^2; U-warps: cross terms, ||u_new||^2)
    // C-warp state (declared here because it is stored after the CTA-wide barrier that follows the role loops)
    double pacc[4][NBLK][2], paccx[4][NUB];
    bool validC[4];
    const int cwC = warp - kFA, grpC = cwC / RSP, rqC = cwC - grpC * RSP;      // 32-sample group, row split
    const int jbC = 32 * grpC;          // lane's samples: jbC + 16 h + 2 gi + e  <->  MMA block mb = 2 h + e, fragment row gi

    if (warp >= kFA + kFC + FU) {
        // =========================================================================== producer warp: the TMA ring
        fused_set_regs<Cfg::LR, Cfg::RU>();
        const char* Ucur_g = f.U + (size_t)ucur * g.uslot_bytes;
        const char* Uprv_g = f.U + (size_t)(ucur ^ 1) * g.uslot_bytes;
        const unsigned rbytes = (unsigned)(g.ldr * 8), ubytes = (unsigned)(g.ldu * 8);
        int s = 0;
        unsigned ph = 0;
        for (int it = 0; it < n_my; ++it) {
            mbar_wait(smem_u32(&ctl->empty[s]), ph ^ 1u);      // the C-warps released tile it - NS
            const long long r0 = ((long long)part + (long long)it * g.n_parts) * TR;
            const int nrows = tile_rows(it);
            const uint32_t full = smem_u32(&ctl->full[s]);
            const uint32_t sb = stages32 + (uint32_t)s * a.stage_bytes;
            if (lane == 0) {
                fence_proxy_async_smem();      // the U-warps wrote the new u into this stage through the generic proxy
                mbar_arrive_expect_tx(full, (unsigned)nrows * (a.pitchX + a.pitchD + rbytes + 2u * ubytes));
            }
            __syncwarp();
            // one bulk copy per matrix: a tile is contiguous in global memory and keeps its row pitch in shared memory (the caller
            // pads the rows of X and d_x so that the pitch is bank-conflict free, see dmf_shape_t)
            if (lane == 0) bulk_g2s(sb, f.X + r0 * (long long)a.pitchX, (unsigned)nrows * a.pitchX, full);
            if (lane == 1) bulk_g2s(sb + a.offD, f.D + r0 * (long long)a.pitchD, (unsigned)nrows * a.pitchD, full);
            if (lane == 2 && K) bulk_g2s(sb + a.offR, f.Rk + r0 * (long long)rbytes, (unsigned)nrows * rbytes, full);
            if (lane == 3) bulk_g2s(sb + a.offU, Ucur_g + r0 * (long long)ubytes, (unsigned)nrows * ubytes, full);
            if (lane == 4) bulk_g2s(sb + a.offUp, Uprv_g + r0 * (long long)ubytes, (unsigned)nrows * ubytes, full);
            __syncwarp();
            if (++s == NS) { s = 0; ph ^= 1u; }
        }
    } else if (warp >= kFA + kFC) {
        // =========================================================================== U-warps: update_u on the row statistics
        fused_set_regs<Cfg::LR, Cfg::RU>();
        const int uw = warp - (kFA + kFC);
        double* Unew_g = reinterpret_cast<double*>(f.U + (size_t)(ucur ^ 2) * g.uslot_bytes);
        double* Unpv_g = reinterpret_cast<double*>(f.U + (size_t)(ucur ^ 3) * g.uslot_bytes);
        const int n2 = a.n_iter2;
        const double l_w = st->l_w;
        const double inv_lw = 1.0 / l_w;       // as u_inner_kernel: reciprocal multiply (<= 1 ulp of a ~1e-4-sized step vs the division of :88)
        const bool at_current = (g.mode == 2);
        const unsigned upitch = (unsigned)(g.ldu * 8);
        const uint32_t beta32 = smem_u32(&ctl->beta[0]);
        // work unit n = (tile n / UP, pass n % UP) goes to U-warp n mod FU: with two unknown types a 32-row tile is two passes of
        // 16 rows x 2 components that two U-warps run side by side (the tile's U latency stays that of one pass)
        for (int n = uw; n < n_my * UP; n += FU) {
            const int it = n / UP, pass = n - it * UP;
            const int s = it % NS;
            const unsigned ph = (unsigned)(it / NS) & 1u;
            // row-statistics buffer of the tile: S = 4 double-buffers (released through sfree), the narrow classes keep one per stage
            const uint32_t stat32 = smem32 + a.offStats + (uint32_t)(Cfg::NSTAT == 2 ? (it & 1) : s) * STATB;
            mbar_wait(smem_u32(&ctl->stats[s]), ph);
            mbar_wait(smem_u32(&ctl->full[s]), ph);        // complete long ago; orders this warp after the bulk copies
            const int nrows = tile_rows(it);
            const long long r0 = ((long long)part + (long long)it * g.n_parts) * TR;
            const uint32_t sb = stages32 + (uint32_t)s * a.stage_bytes;
            if constexpr (NUB == 2) {
                // lane = (row, component): 16 rows of the tile in both half warps, component q = lane / 16
                const int row = 16 * pass + (lane & 15), q = lane >> 4;
                const bool live = row < nrows;
                double v[NG];
#pragma unroll
                for (int i = 0; i < NG; ++i) v[i] = 0.0;
                {
                    const uint32_t sbase = stat32 + (uint32_t)row * (NG * 8u);
#pragma unroll
                    for (int w = 0; w < SG; ++w)
#pragma unroll
                        for (int i = 0; i < NG; ++i) {
                            double t;
                            lds1(sbase + (uint32_t)w * (TR * NG * 8u) + (uint32_t)i * 8u, t);
                            v[i] += t;
                        }
                    if constexpr (Cfg::NSTAT == 2) {
                        __syncwarp();
                        if (lane == 0) mbar_arrive(smem_u32(&ctl->sfree[it & 1]));
                    }
                }
                double cu, pv, cuo;
                lds1(sb + a.offU + (uint32_t)row * upitch + (uint32_t)q * 8u, cu);
                lds1(sb + a.offUp + (uint32_t)row * upitch + (uint32_t)q * 8u, pv);
                lds1(sb + a.offU + (uint32_t)row * upitch + (uint32_t)(q ^ 1) * 8u, cuo);
                if (live && q == 0) {      // cost of the incoming iterate: -2 u^T b + u^T H u of this row
                    double ct = cu * (fma(v[3], cuo, v[2] * cu) - 2.0 * v[0]);
                    ct = fma(cuo, fma(v[4], cuo, v[3] * cu) - 2.0 * v[1], ct);
                    cost += ct;
                }
#ifndef DMF_SKIP_U
                {
                    const double c = (q ? v[1] : v[0]) * inv_lw, mh_own = (q ? v[4] : v[2]) * inv_lw, mh_oth = v[3] * inv_lw;
                    const double am_own = at_current ? -mh_own : 1.0 - mh_own, am_oth = -mh_oth;
                    const bool tame = fabs(c) < 1e150 && fabs(mh_own) < 1e150 && fabs(mh_oth) < 1e150 && fabs(cu) <= 1.0 && fabs(pv) <= 1.0;
                    if (__all_sync(0xffffffffu, tame)) {
                        if (at_current) fused_u_loop_split<true, true>(cu, pv, am_own, am_oth, c, beta32, n2);
                        else fused_u_loop_split<false, true>(cu, pv, am_own, am_oth, c, beta32, n2);
                    } else {
                        if (at_current) fused_u_loop_split<true, false>(cu, pv, am_own, am_oth, c, beta32, n2);
                        else fused_u_loop_split<false, false>(cu, pv, am_own, am_oth, c, beta32, n2);
                    }
                }
#endif
                if (live) {
                    Unew_g[(size_t)(r0 + row) * g.ldu + q] = cu;
                    Unpv_g[(size_t)(r0 + row) * g.ldu + q] = pv;
                    ssq = fma(cu, cu, ssq);
                }
                {
                    const double un = live ? cu : 0.0;
                    asm volatile("st.shared.f64 [%0], %1;" ::"r"(sb + a.offU + (uint32_t)row * upitch + (uint32_t)q * 8u), "d"(un) : "memory");
                }
            } else {
            const bool live = lane < nrows;
            const int row = lane < TR ? lane : 0;
            // row statistics: the 4 sample-group partials in group order; the buffer is free for tile it + 2 as soon as they are in registers
            double v[NG];
#pragma unroll
            for (int i = 0; i < NG; ++i) v[i] = 0.0;
            {
                const uint32_t sbase = stat32 + (uint32_t)row * (NG * 8u);
#pragma unroll
                for (int w = 0; w < SG; ++w)
#pragma unroll
                    for (int i = 0; i < NG; ++i) {
                        double t;
                        lds1(sbase + (uint32_t)w * (TR * NG * 8u) + (uint32_t)i * 8u, t);
                        v[i] += t;
                    }
                if constexpr (Cfg::NSTAT == 2) {
                    __syncwarp();
                    if (lane == 0) mbar_arrive(smem_u32(&ctl->sfree[it & 1]));
                }
            }
            double u[NUB], up[NUB];
#pragma unroll
            for (int q = 0; q < NUB; ++q) {
                lds1(sb + a.offU + (uint32_t)row * upitch + (uint32_t)q * 8u, u[q]);
                lds1(sb + a.offUp + (uint32_t)row * upitch + (uint32_t)q * 8u, up[q]);
            }
            if (live) {      // cost of the incoming iterate: -2 u^T b + u^T H u of this row (rowgram4_kernel, writer lanes)
                double ct = 0.0;
#pragma unroll
                for (int q = 0; q < NUB; ++q) {
                    double hq = 0.0;
#pragma unroll
                    for (int q2 = 0; q2 < NUB; ++q2) hq = fma(v[NUB + (q <= q2 ? tri_index(q, q2, NUB) : tri_index(q2, q, NUB))], u[q2], hq);
                    ct = fma(u[q], hq - 2.0 * v[q], ct);
                }
                cost += ct;
            }
#ifndef DMF_SKIP_U
            if (at_current) fused_u_iterate<true, NUB>(u, up, v, beta32, n2, inv_lw);
            else fused_u_iterate<false, NUB>(u, up, v, beta32, n2, inv_lw);
#endif
            // new iterate: global (other slot pair) and the stage (the C-warps form u (x) [R_trunc | u] and bx_u from it)
            if (live) {
#pragma unroll
                for (int q = 0; q < NUB; ++q) {
                    if (q < g.nu) {
                        Unew_g[(size_t)(r0 + lane) * g.ldu + q] = u[q];
                        Unpv_g[(size_t)(r0 + lane) * g.ldu + q] = up[q];
                        ssq = fma(u[q], u[q], ssq);
                    }
                }
            }
            if (lane < TR) {
#pragma unroll
                for (int q = 0; q < NUB; ++q) {
                    const double un = (live && q < g.nu) ? u[q] : 0.0;
                    asm volatile("st.shared.f64 [%0], %1;" ::"r"(sb + a.offU + (uint32_t)lane * upitch + (uint32_t)q * 8u), "d"(un) : "memory");
                }
            }
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&ctl->udone[s]));
        }
    } else if (warp < kFA) {
        // =========================================================================== A-warps: row statistics
        fused_set_regs<Cfg::LR, Cfg::RA>();
        const int arb = warp % Cfg::RB, asg = warp / Cfg::RB;       // row block of the tile, sample group
        const int rowA = 8 * arb + (gi >> 1) + 4 * (gi & 1);        // fragment row gi <-> tile row: lanes of a quarter warp read rows 4 apart
        const int blk0 = asg * NSB;                                 // the warp's first block of 8 samples
        const int nblk = min(NSB, max(0, (N + 7) / 8 - blk0));      // blocks that exist
        const bool cols_full = 8 * (blk0 + NSB) <= N;               // every sample of this warp exists: no column masks
        const int jlane = 8 * blk0 + 2 * ti;
        double nab[NSB][KS > 0 ? KS : 1];                           // B operand: -alpha_k[4 kk + ti][sample gi of block sb]
#pragma unroll
        for (int sb = 0; sb < NSB; ++sb) {
            const int j = 8 * (blk0 + sb) + gi;
#pragma unroll
            for (int kk = 0; kk < (KS > 0 ? KS : 1); ++kk) {
                const int k = 4 * kk + ti;
                nab[sb][kk] = (KS > 0 && j < N && k < K) ? -Acur[(size_t)k * N + j] : 0.0;
            }
        }
        const unsigned rpitch = (unsigned)(g.ldr * 8);
        const uint32_t xrel = (uint32_t)rowA * a.pitchX + (uint32_t)jlane * 8u;
        const uint32_t drel = a.offD + (uint32_t)rowA * a.pitchD + (uint32_t)jlane * (unsigned)sizeof(WT);
        const uint32_t ta = smem32 + a.offTab + (uint32_t)(4 * blk0 + ti) * PAIRB;
        const uint32_t srel = a.offStats + (uint32_t)asg * (TR * NG * 8u) + (uint32_t)rowA * (NG * 8u);
        int s = 0;
        unsigned ph = 0;
        uint32_t sb32 = stages32;
        const bool writer = (ti == 0);
        for (int it = 0; it < n_my; ++it) {
            mbar_wait(smem_u32(&ctl->full[s]), ph);
            const int nrows = tile_rows(it);
            double rfrag[KS > 0 ? KS : 1];                          // A operand: R_trunc[row][4 kk + ti]
#pragma unroll
            for (int kk = 0; kk < KS; ++kk) {
                const int k = 4 * kk + ti;
                double t = 0.0;
                if (k < K) lds1(sb32 + a.offR + (uint32_t)rowA * rpitch + (uint32_t)k * 8u, t);
                rfrag[kk] = t;
            }
            double acc[NG];
#pragma unroll
            for (int i = 0; i < NG; ++i) acc[i] = 0.0;
#ifndef DMF_SKIP_A
            if (cols_full && nrows == TR) fused_row_stats<false, WT, KS, NUB, NSB>(sb32 + xrel, sb32 + drel, ta, rfrag, nab, nblk, jlane, N, true, cost, acc);
            else fused_row_stats<true, WT, KS, NUB, NSB>(sb32 + xrel, sb32 + drel, ta, rfrag, nab, nblk, jlane, N, rowA < nrows, cost, acc);
#endif
            // sum over the 4 lanes of the row (ti), then one partial per (sample group, row, value)
#pragma unroll
            for (int i = 0; i < NG; ++i) {
                acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 1);
                acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], 2);
            }
            if constexpr (Cfg::NSTAT == 2) {
                if (it >= 2) mbar_wait(smem_u32(&ctl->sfree[it & 1]), ((unsigned)((it >> 1) - 1)) & 1u);     // tile it - 2's partials were read
            }
            {   // the 8 lanes with ti == 0 store their row's record and arrive themselves (no warp-wide reconvergence)
                const uint32_t sbase = smem32 + srel + (uint32_t)(Cfg::NSTAT == 2 ? (it & 1) : s) * STATB;
#pragma unroll
                for (int i = 0; i < NG; ++i)
                    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %2, 0;\n@p st.shared.f64 [%0], %1;\n}" ::"r"(sbase + (uint32_t)i * 8u), "d"(acc[i]), "r"((unsigned)writer) : "memory");
                asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %1, 0;\n@p mbarrier.arrive.shared::cta.b64 _, [%0];\n}" ::"r"(smem_u32(&ctl->stats[s])), "r"((unsigned)writer) : "memory");
            }
            sb32 += a.stage_bytes;
            if (++s == NS) { s = 0; ph ^= 1u; sb32 = stages32; }
        }
    } else {
        // =========================================================================== C-warps: Gram panel with the new u
        fused_set_regs<Cfg::LR, Cfg::RC>();
#pragma unroll
        for (int mb = 0; mb < 4; ++mb) {
            validC[mb] = jbC + 16 * (mb >> 1) + 2 * gi + (mb & 1) < N;
#pragma unroll
            for (int nb = 0; nb < NBLK; ++nb) { pacc[mb][nb][0] = 0.0; pacc[mb][nb][1] = 0.0; }
#pragma unroll
            for (int q = 0; q < NUB; ++q) paccx[mb][q] = 0.0;
        }
        const unsigned upitch = (unsigned)(g.ldu * 8), rpitch = (unsigned)(g.ldr * 8);
        // B operand of the panel MMA: u_q times the lane's entry of W = [R_trunc | u] (column 8 wb + gi), read from the stage
        // (the U-warp left the new u there); a column that does not exist reads a zero (pitch 0: no select in the loop)
        unsigned w_off[WB], w_pitch[WB];
#pragma unroll
        for (int wb = 0; wb < WB; ++wb) {
            const int w = 8 * wb + gi;
            const bool isr = w < KB, exists = isr ? w < K : (w - KB) < g.nu && (w - KB) < NUB;
            w_off[wb] = !exists ? a.zero_off : (isr ? a.offR + (unsigned)w * 8u : a.offU + (unsigned)(w - KB) * 8u);
            w_pitch[wb] = !exists ? 0u : (isr ? rpitch : upitch);
        }
        const bool work = jbC < N;                     // (else this sample group is empty, the warp only keeps the ring moving)
        const bool cols_full = jbC + 32 <= N;
        const uint32_t xoff = (uint32_t)(jbC + 2 * gi) * 8u, doff = (uint32_t)(jbC + 2 * gi) * (unsigned)sizeof(WT);
        const int ks0 = rqC * KSW;
        int s = 0;
        unsigned ph = 0;
        uint32_t sb32 = stages32;
        for (int it = 0; it < n_my; ++it) {
            mbar_wait(smem_u32(&ctl->udone[s]), ph);
            mbar_wait(smem_u32(&ctl->full[s]), ph);
            const int nrows = tile_rows(it);
#ifndef DMF_SKIP_C
            if (work) {
                if (cols_full && nrows == TR) fused_panel_tile<false, WT, NUB, KSW, WB>(a, sb32, nrows, ti, ks0, xoff, doff, w_off, w_pitch, validC, pacc, paccx);
                else fused_panel_tile<true, WT, NUB, KSW, WB>(a, sb32, nrows, ti, ks0, xoff, doff, w_off, w_pitch, validC, pacc, paccx);
            }
#endif
            __syncwarp();
            if (lane == 0) mbar_arrive(smem_u32(&ctl->empty[s]));
            sb32 += a.stage_bytes;
            if (++s == NS) { s = 0; ph ^= 1u; sb32 = stages32; }
        }
    }
    __syncthreads();
    // CTA record: [cost, ||u||^2, panel NCOL x N, bx NUB x N] - the stage ring is free once every role left its loop.  The RSP
    // C-warps that share a sample group (row splits of the tile) add their sums in split order.
    {
        double* rec = reinterpret_cast<double*>(smem + kFusedCtlBytes);
#pragma unroll
        for (int r = 0; r < RSP; ++r) {
            if (warp >= kFA && warp < kFA + kFC && rqC == r) {
#pragma unroll
                for (int mb = 0; mb < 4; ++mb) {
                    const int j = jbC + 16 * (mb >> 1) + 2 * gi + (mb & 1);
#pragma unroll
                    for (int nb = 0; nb < NBLK; ++nb)
#pragma unroll
                        for (int e = 0; e < 2; ++e) {
                            // block nb = q WB + wb holds u_q W[8 wb + 2 ti + e]: W columns < KB are R_trunc, then u_q2 (upper triangle kept)
                            const int q = nb / WB, w = 8 * (nb - q * WB) + 2 * ti + e, q2 = w - KB;
                            int c = -1;
                            if (w < KB) c = q * KB + w;
                            else if (q2 >= q && q2 < NUB) c = NUB * KB + tri_index(q < NUB ? q : 0, q2 >= q ? q2 : q, NUB);
                            if (validC[mb] && c >= 0) {
                                double* p = &rec[2 + (size_t)c * N + j];
                                *p = (r == 0) ? pacc[mb][nb][e] : *p + pacc[mb][nb][e];
                            }
                        }
#pragma unroll
                    for (int q = 0; q < NUB; ++q) {
                        double t = paccx[mb][q];
                        t += __shfl_xor_sync(0xffffffffu, t, 1);
                        t += __shfl_xor_sync(0xffffffffu, t, 2);
                        if (validC[mb] && ti == 0) {
                            double* p = &rec[2 + (size_t)(NCOL + q) * N + j];
                            *p = (r == 0) ? t : *p + t;
                        }
                    }
                }
            }
            if (r + 1 < RSP) __syncthreads();
        }
    }
    // scalar partials: warp sums, then the warps in order
    {
        double c = cost, q = ssq;
#pragma unroll
        for (int o = 16; o >= 1; o >>= 1) {
            c += __shfl_xor_sync(0xffffffffu, c, o);
            q += __shfl_xor_sync(0xffffffffu, q, o);
        }
        if (lane == 0) { ctl->wsum[0][warp] = c; ctl->wsum[1][warp] = q; }
    }
    __syncthreads();
    double* rec = reinterpret_cast<double*>(smem + kFusedCtlBytes);
    if (tid == 0) {
        double c = 0.0, q = 0.0;
        for (int w = 0; w < Cfg::WARPS; ++w) { c += ctl->wsum[0][w]; q += ctl->wsum[1][w]; }
        rec[0] = c;
        rec[1] = q;
    }
    __syncthreads();
    const int n = 2 + (NCOL + NUB) * N;
    {
        double* p = f.part + (size_t)part * g.part_stride;
        for (int e = tid; e < n; e += THREADS) p[e] = rec[e];
    }
    if (!hier_reduce(g, f, f.red, n, &ctl->flag)) return;
    __threadfence();
    __syncthreads();
    // ------------------------------------------------------------------------------- last CTA of the fit: test, then commit
    if (tid == 0) {
        const double cf = f.red[0], su = f.red[1];
        int commit = 1;
        if (a.flags & kFlagPartial) {
            // CpG rows sharded over GPUs: publish this GPU's sums; alpha_inner_kernel tests and commits on the all-reduced sums
            f.scal[0] = cf;
            f.scal[4] = su;
        } else {
            // a phase-1 iterate closes an outer iteration; a stop leaves the pass uncommitted
            if (st->phase == 1 && state_close_outer(st, f, cf, a.tol)) commit = 0;
            if (commit) {
                const int t0 = st->t_u, n2 = a.n_iter2;
                st->u_cur = ucur ^ 2;
                state_end_u(st, a.mom_a[t0 + n2], t0 + n2, st->l_w, n2 > 0);
                state_u_norm(st, su);
                st->phase = 1;
            }
        }
        ctl->commit = commit;
    }
    __syncthreads();
    if (!ctl->commit) return;
    for (int e = tid; e < (NCOL + NUB) * N; e += THREADS) {
        const int c = e / N, j = e - c * N;
        const double v = f.red[2 + e];
        if (c >= NCOL) {
            const int q = c - NCOL;
            if (q < g.nu) f.gbx[(size_t)(K + q) * N + j] = v;
        } else if (c < NUB * KB) {
            const int q = c / KB, k = c - q * KB;
            if (q < g.nu && k < K) {
                f.gram[((size_t)(K + q) * g.Kt + k) * N + j] = v;
                f.gram[((size_t)k * g.Kt + (K + q)) * N + j] = v;
            }
        } else {
            int e2 = c - NUB * KB, q = 0;
            while (e2 >= NUB - q) { e2 -= NUB - q; ++q; }
            const int q2 = q + e2;
            if (q2 < g.nu) {
                f.gram[((size_t)(K + q) * g.Kt + (K + q2)) * N + j] = v;
                f.gram[((size_t)(K + q2) * g.Kt + (K + q)) * N + j] = v;
            }
        }
    }
}

}  // namespace dmf
