// dmf_device.cuh — device-side building blocks shared by the sm_100a deconvolution kernels:
// mbarrier / bulk-copy (TMA, UBLKCP) wrappers, the producer-warp tile pipeline, and the
// deterministic two-level cross-CTA reduction ("last CTA of a group, last group of the fit").
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace dmf {

constexpr int kConsumers = 256;             // threads per CTA: 8 warps, all compute; warp 0 also feeds the TMA ring
constexpr int kThreads = kConsumers;
constexpr int kStages = 5;                  // smem ring depth (kStages - 2 tiles requested ahead)
constexpr int kGroup = 16;                  // CTAs per first-level reduction group
constexpr int kMaxSrc = 5;                  // matrices streamed per stage: X, D, Rk, U, Uprev
constexpr int kMaxKt = 32;                  // K + n_u supported by the register-tiled kernels
constexpr int kMaxSamples = 2 * kConsumers; // N supported (make_plan: N <= kConsumers x columns per thread, at most 2)

// ------------------------------------------------------------------------------------------------
// Device-side descriptors (mirrors of the host structs in dmf_api.cu)
struct FitState {
    double a1, a2;                 // extrapolation scalars (deconvolution.py:84,96)
    double l_w, l_w_old;           // ||alpha_unk||^2 * dmax^2 and its previous value
    double l_h, l_h_old;           // ||R||^2 * dmax^2 and its previous value
    double cf, cf_prev;            // cost after / before the last outer iteration
    double dmax, dmax2;            // max d_x and its square
    double ssq_rk, ssq_u;          // ||R_trunc||_F^2 (constant) and ||u||_F^2 (current)
    int u_cur, a_cur;              // ping-pong slots holding the current iterate
    int n_outer, done;             // done: 0 running, 1 converged, 3 numerical failure (NaN in projection)
    int t_u, t_a;                  // inner iterations of update_u / update_alpha executed so far (index into the momentum table)
    int phase;                     // fused engine: 1 = the cost of the current iterate has not been evaluated yet (dmf_fused.cuh)
    int pad;
};

struct FitDev {
    const char* X;
    const char* D;
    const char* Rk;
    const int32_t* rows;
    char* U;
    char* A;
    const double* purity;
    double* trace;
    double* part;        // [n_parts][part_stride] per-CTA partial sums
    double* gpart;       // [n_groups][part_stride] per-group partial sums
    unsigned* tickets;   // [n_groups + 1]
    FitState* st;
    double* rowgram;     // Gram engine: [M][warps per row][NG] per-row statistics of the U step
    double* gram;        // Gram engine: [Kt][Kt][N] per-sample G_j = R^T diag(d_.j) R      (written by gram_panel_kernel: this GPU's rows);
                         // stream engine, row-sharded: [Kt][N] this GPU's alpha gradient (alpha_pass_kernel)
    double* gbx;         // Gram engine: [Kt][N]     per-sample R^T (d_.j o x_.j)
    double* scal;        // Gram engine: [8] row-sharded runs: this GPU's [cost, ||R_trunc||^2, ||u||^2 (set-up), max d, ||u||^2 (U step)]
    double* rgram;       // what alpha_inner_kernel / finalize_cost_kernel READ: == gram / gbx / scal on one GPU, the all-reduced
    double* rgbx;        //   copies when the CpG rows are sharded over several GPUs
    double* rscal;
    double* red;         // Gram engine: [part_stride] totals of the last cross-CTA reduction
    // bootstrap resamples in multiplicity form: the fit's rows are the SOURCE rows of the shared X, d_x, R_trunc; source row m
    // was drawn mult[m] times and owns the u rows offs[m] .. offs[m + 1] (positions sorted by source row)
    const int32_t* mult;
    const int32_t* offs;
    const int32_t* pos_row;   // source row of every position (nondecreasing)
    double* usum;        // [M][NG] per source row: sum of u over its positions, then the upper triangle of sum u u^T
    int trace_cap;
    int pad;
};

struct Geom {
    long long M;
    int N, K, nu, Kt;
    long long ldx, ldd, ldr, ldu;  // row pitches in elements (all even, zero padded)
    int Kp, nup;                   // K and n_u rounded up to even: columns actually loaded
    int rpt;                       // rows per thread per tile in the U pass (tile_rows = rpt * rows-groups)
    long long uslot_bytes;         // bytes between the two U slots
    int tile_rows, n_tiles;
    int ntc, rg;                   // threads per row (power of two), row groups per CTA
    int n_parts, n_groups;         // CTAs per fit, reduction groups per fit
    int part_stride;               // doubles per partial record
    unsigned offX, offD, offR, offU, offUp, stage_bytes;   // smem stage layout (bytes)
    unsigned row_bulk;             // bit0 X, bit1 D, bit2 Rk: per-row bulk copies legal in gather mode
    unsigned tile_tx[kMaxSrc];     // bytes of one FULL tile of X, D, Rk, U, Uprev (each a multiple of 16)
    int mode;                      // DMF_MODE_*
    int gather;                    // any fit uses a row index
    int fit_major;                 // grid = (fits, parts) instead of (parts, fits): CTAs that run together work on the SAME row
                                   // tiles of different fits, so fits sharing X / d_x / R_trunc are served from L2
    int multmode;                  // fits are bootstrap resamples in multiplicity form (FitDev::mult / offs / usum)
    int stages;                    // depth of the shared-memory ring actually used (3 .. kStages); 0 = kStages
};
__device__ __forceinline__ int n_stages(const Geom& g) { return g.stages ? g.stages : kStages; }
__device__ __forceinline__ int part_id(const Geom& g) { return g.fit_major ? (int)blockIdx.y : (int)blockIdx.x; }
__device__ __forceinline__ int fit_id(const Geom& g) { return g.fit_major ? (int)blockIdx.x : (int)blockIdx.y; }

// ------------------------------------------------------------------------------------------------
// kernel argument block and shared-memory control block
struct PassArgs {
    Geom g;
    const FitDev* fits;
    int k_inner;      // Frank-Wolfe iteration index (reference-shaped pass) / n_iter2 (Gram-engine inner kernels)
    int flags;        // kFlag*
    double tol;
    int ca0, cb0;     // gram_panel_kernel: first chunk (pair of padded register-row entries) of the za / zb blocks
    int with_x;       // gram_panel_kernel: also emit R^T (d o x) for the za block
    int pad;
    // momentum table (data independent, deconvolution.py:83-85): mom_a[t] = a_t (a_0 = 1, a_{t+1} = (1 + sqrt(1 + 4 a_t^2)) / 2),
    // mom_m[t] = (a_t - 1) / a_{t+1}; filled by the host for every inner-iteration index a launch can reach
    const double* mom_a;
    const double* mom_m;
};
constexpr int kFlagInitial = 1;   // init_cost_kernel: set-up pass (norms, max d, no termination test)
constexpr int kFlagFW = 2;        // alpha_pass_kernel: Frank-Wolfe step instead of projected gradient
constexpr int kFlagPartial = 4;   // CpG rows sharded over GPUs: publish this GPU's sums to FitDev::scal (and gram), leave the state to
                                  // finalize_cost_kernel / alpha_inner_kernel (Gram engine) or u_commit_kernel / alpha_commit_kernel
                                  // (stream engine), which run on the all-reduced sums
constexpr int kFlagF32 = 8;       // finalize_cost_kernel, alpha_commit_kernel: alpha is stored as float
constexpr int kFlagFusedCommit = 16;   // alpha_inner_kernel after a kFlagPartial fused pass (row-sharded): run the termination test and commit
                                       // the U step on the all-reduced sums (what the fused pass's last CTA does on one GPU)

struct TileSrc {
    const char* base;      // global base of the matrix (fit-specific), nullptr = absent
    long long pitch;       // bytes per row
    unsigned off;          // offset inside the stage
    unsigned char gathered;   // rows come through the fit's row index
    unsigned char row_bulk;   // per-row bulk copy legal (pitch % 16 == 0)
    unsigned short pad;
};
struct SmemCtl {
    unsigned long long full[kStages];
    unsigned long long empty[kStages];
    TileSrc src[kMaxSrc];   // what one stage is made of (written once by thread 0)
    int flag;
    int pad;
};
constexpr unsigned kCtlBytes = 256;
static_assert(sizeof(SmemCtl) <= kCtlBytes, "control block too large");

// ------------------------------------------------------------------------------------------------
// PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}
// 1-D bulk asynchronous copy global -> shared (TMA engine, SASS UBLKCP); 16-byte aligned, size % 16 == 0
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                 "l"(src), "r"(bytes), "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void consumer_bar() { asm volatile("bar.sync 1, %0;" ::"n"(kConsumers) : "memory"); }

// ------------------------------------------------------------------------------------------------
// Tile pipeline.  One stage holds `tile_rows` rows of X, D, Rk, U(cur) and optionally U(prev).

// Executed by the whole producer warp.  Fills stage `sbase` with rows [r0, r0+nrows) of every source
// and arms `full_bar` with the number of bytes that will arrive asynchronously.
__device__ __forceinline__ void produce_tile(const TileSrc* src, int nsrc, const int32_t* rows, long long r0, int nrows,
                                             char* sbase, uint32_t full_bar, int lane) {
    uint32_t tx = 0;
    // pass 1: everything that cannot go through the bulk-copy engine is copied by the warp itself
    for (int s = 0; s < nsrc; ++s) {
        const TileSrc& m = src[s];
        if (m.base == nullptr) continue;
        char* dst = sbase + m.off;
        if (m.gathered && rows != nullptr) {
            if (m.row_bulk) {
                tx += (uint32_t)(nrows * m.pitch);
            } else {
                for (int r = 0; r < nrows; ++r) {
                    const char* g = m.base + (long long)rows[r0 + r] * m.pitch;
                    for (long long b = lane; b < m.pitch; b += 32) dst[r * m.pitch + b] = g[b];
                }
            }
        } else {
            const long long total = (long long)nrows * m.pitch;
            const long long bulk = total & ~15LL;
            tx += (uint32_t)bulk;
            const char* g = m.base + r0 * m.pitch;
            for (long long b = bulk + lane; b < total; b += 32) dst[b] = g[b];
        }
    }
    __syncwarp();
    if (lane == 0) mbar_arrive_expect_tx(full_bar, tx);
    __syncwarp();
    // pass 2: issue the bulk copies
    for (int s = 0; s < nsrc; ++s) {
        const TileSrc& m = src[s];
        if (m.base == nullptr) continue;
        const uint32_t dst = smem_u32(sbase + m.off);
        if (m.gathered && rows != nullptr) {
            if (m.row_bulk) {
                for (int r = lane; r < nrows; r += 32)
                    bulk_g2s(dst + (uint32_t)(r * m.pitch), m.base + (long long)rows[r0 + r] * m.pitch, (uint32_t)m.pitch,
                             full_bar);
            }
        } else if (lane == 0) {
            const long long bulk = ((long long)nrows * m.pitch) & ~15LL;
            // one copy may not exceed the mbarrier tx-count range comfortably; chunk at 64 KB
            const char* g = m.base + r0 * m.pitch;
            for (long long o = 0; o < bulk; o += 65536) {
                const uint32_t n = (uint32_t)((bulk - o) < 65536 ? (bulk - o) : 65536);
                bulk_g2s(dst + (uint32_t)o, g + o, n, full_bar);
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Deterministic two-level reduction of per-CTA partial records.
// Every CTA of the fit has written `n` doubles to f.part[blockIdx.x * stride ...].  Returns true in
// exactly one CTA of the fit, in which out_sm[0..n) holds the totals, summed in CTA-index order
// inside each group and in group order across groups (independent of arrival order).
__device__ __forceinline__ bool hier_reduce(const Geom& g, const FitDev& f, double* out_sm, int n, int* s_flag) {
    const int tid = threadIdx.x;
    const int grp = part_id(g) / kGroup;
    const int gfirst = grp * kGroup;
    const int gsize = min(kGroup, g.n_parts - gfirst);
    __threadfence();
    __syncthreads();
    if (tid == 0) *s_flag = (atomicAdd(&f.tickets[grp], 1u) == (unsigned)(gsize - 1));
    __syncthreads();
    if (!*s_flag) return false;
    __threadfence();
    const bool single = (g.n_groups == 1);
    for (int e = tid; e < n; e += blockDim.x) {
        // the group's records in CTA order; the loads are issued together (one L2 round trip per element instead of gsize)
        double v[kGroup];
#pragma unroll
        for (int p = 0; p < kGroup; ++p) v[p] = p < gsize ? __ldcg(&f.part[(size_t)(gfirst + p) * g.part_stride + e]) : 0.0;
        double s = 0.0;
#pragma unroll
        for (int p = 0; p < kGroup; ++p) s += v[p];
        if (single)
            out_sm[e] = s;
        else
            f.gpart[(size_t)grp * g.part_stride + e] = s;
    }
    if (tid == 0) f.tickets[grp] = 0u;   // re-arm for the next launch
    if (single) {
        __syncthreads();
        return true;
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) *s_flag = (atomicAdd(&f.tickets[g.n_groups], 1u) == (unsigned)(g.n_groups - 1));
    __syncthreads();
    if (!*s_flag) return false;
    __threadfence();
    for (int e = tid; e < n; e += blockDim.x) {
        double s = 0.0;
        for (int q0 = 0; q0 < g.n_groups; q0 += kGroup) {      // group records in group order, kGroup loads in flight
            double v[kGroup];
#pragma unroll
            for (int q = 0; q < kGroup; ++q) v[q] = q0 + q < g.n_groups ? __ldcg(&f.gpart[(size_t)(q0 + q) * g.part_stride + e]) : 0.0;
#pragma unroll
            for (int q = 0; q < kGroup; ++q) s += v[q];
        }
        out_sm[e] = s;
    }
    if (tid == 0) f.tickets[g.n_groups] = 0u;
    __syncthreads();
    return true;
}

// extrapolation weight of the accelerated projected-gradient steps (deconvolution.py:83-85, 95-97)
__device__ __forceinline__ double next_momentum(double a_prev) { return (1.0 + sqrt(1.0 + 4.0 * a_prev * a_prev)) / 2.0; }
__device__ __forceinline__ double extrap_beta(double a_prev, double a_next, double l_old, double l_new) {
    return fmin((a_prev - 1.0) / a_next, 0.9999 * sqrt(l_old / l_new));
}

// ------------------------------------------------------------------------------------------------
// The reference's outer-loop bookkeeping (deconvolution.py:192-221), written once for every engine.  Each function runs in the
// one thread that owns the fit state; the outer-iteration counts of the parity tests depend on every operation and its order.
// The set-up reads its partial record through a pointer and the close returns `done`: in those shapes ptxas allocates the
// calling kernels exactly as it did for the inline copies these functions replace.

// l_w / l_h (deconvolution.py:192-204, :212, :216): the Frobenius norm, squared, times max(d_x)^2
__device__ __forceinline__ double lipschitz(double ssq, double dmax2) {
    const double nrm = sqrt(ssq);
    return (nrm * nrm) * dmax2;
}
// max d_x over the CTA partial records [cost, ssq_rk, ssq_u, dmax] (a max, not a sum: hier_reduce does not carry it)
__device__ __forceinline__ double part_dmax(const Geom& g, const FitDev& f) {
    double dm = 0.0;
    for (int p = 0; p < g.n_parts; ++p) dm = fmax(dm, __ldcg(&f.part[(size_t)p * g.part_stride + 3]));
    return dm;
}
// ||alpha[-n_u:]||_F^2 of the alpha slot A (deconvolution.py:198): tiny, done serially in row-major order
template <typename T>
__device__ __forceinline__ double alpha_unk_ssq(const Geom& g, const T* A) {
    double sa = 0.0;
    for (int q = 0; q < g.nu; ++q)
        for (int j = 0; j < g.N; ++j) {
            const double v = (double)A[(size_t)(g.K + q) * g.N + j];
            sa = fma(v, v, sa);
        }
    return sa;
}

// set-up (deconvolution.py:192-204) from the record [cost, ||R_trunc||^2, ||u||^2] of the initial iterate, max d_x and its alpha slot A
template <typename T>
__device__ __forceinline__ void state_setup(FitState* st, const FitDev& f, const double* rec, double dmax, const Geom& g, const T* A) {
    const double cf = rec[0];
    st->dmax = dmax;
    st->dmax2 = dmax * dmax;
    st->ssq_rk = rec[1];
    st->ssq_u = rec[2];
    st->l_w = lipschitz(alpha_unk_ssq(g, A), st->dmax2);
    st->l_w_old = st->l_w;
    st->l_h = lipschitz(rec[1] + rec[2], st->dmax2);
    st->l_h_old = st->l_h;
    st->a1 = 1.0;
    st->a2 = 1.0;
    st->cf = cf;
    st->cf_prev = cf;
    st->n_outer = 0;
    st->t_u = 0;
    st->t_a = 0;
    st->phase = 0;
    if (f.trace && f.trace_cap > 0) f.trace[0] = cf;
}

// termination test (deconvolution.py:220), plus a NaN cost
__device__ __forceinline__ bool outer_stops(double cf, double cf_prev, double tol) { return fabs(cf - cf_prev) < tol || !(cf == cf); }

// close of an outer iteration (deconvolution.py:218-221) with the cost of the new iterate; a stop sets done = 1 (converged) or
// 3 (NaN cost).  Returns whether the fit is done.
__device__ __forceinline__ bool state_close_outer(FitState* st, const FitDev& f, double cf, double tol) {
    const double prev = st->cf;
    st->cf_prev = prev;
    st->cf = cf;
    const int n = st->n_outer + 1;
    st->n_outer = n;
    if (f.trace && n < f.trace_cap) f.trace[n] = cf;
    st->phase = 0;                                  // the cost of the current iterate is known (dmf_fused.cuh)
    if (outer_stops(cf, prev, tol)) st->done = (cf == cf) ? 1 : 3;
    return st->done != 0;
}

// end of the U step (deconvolution.py:84-89): momentum a1 and inner-iteration index; l_w_ = l_w once a step ran
__device__ __forceinline__ void state_end_u(FitState* st, double a1_next, int t_u_next, double l_w_stepped, bool stepped) {
    st->a1 = a1_next;
    st->t_u = t_u_next;
    if (stepped) st->l_w_old = l_w_stepped;
}
// ||u||^2 after the U step and l_h = ||[R_trunc, u]||^2 dmax^2 (deconvolution.py:212, read by the alpha steps only)
__device__ __forceinline__ void state_u_norm(FitState* st, double ssq_u) {
    st->ssq_u = ssq_u;
    st->l_h = lipschitz(st->ssq_rk + ssq_u, st->dmax2);
}

// end of the alpha step (deconvolution.py:96-101, :216 / :327): l_w from ||alpha[-n_u:]||^2; the projected-gradient step also
// advances its momentum a2 and inner-iteration index, and l_h_ = l_h once a step ran (Frank-Wolfe has no momentum)
__device__ __forceinline__ void state_end_alpha(FitState* st, double ssq_alpha_unk, bool projected_gradient, double a2_next,
                                                int t_a_next, double l_h_stepped, bool stepped) {
    st->l_w = lipschitz(ssq_alpha_unk, st->dmax2);
    if (projected_gradient) {
        st->a2 = a2_next;
        st->t_a = t_a_next;
        if (stepped) st->l_h_old = l_h_stepped;
    }
}

}  // namespace dmf
