// dmf_api.cu — extern "C" surface of libdemethify_sm100.so (see include/demethify_b200.h).
// Host logic only: shape validation, launch geometry, kernel dispatch, the outer-loop driver.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/demethify_b200.h"
#include "dmf_device.cuh"
#include "dmf_inst.h"
#include "dmf_gram.cuh"
#include "dmf_fused.cuh"
#include "dmf_rng.cuh"

using namespace dmf;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
    g_err = msg;
    return code;
}
#define CUDA_TRY(expr)                                                                                      \
    do {                                                                                                    \
        cudaError_t e__ = (expr);                                                                           \
        if (e__ != cudaSuccess) return fail(DMF_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e__)); \
    } while (0)

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

}  // namespace

struct dmf_handle_s {
    int device;
    int sm_count;
    int max_smem_optin;
};

namespace {

// ---------------------------------------------------------------------------------------------
// kernel tables: the template instantiations live in dmf_inst_*.cu (one translation unit per storage-type pair)
kern_t by_types(const dmf_shape_t& s, kern_t (*f[4])(int, int, int), int a, int b, int c) {
    const int i = (s.dtype == DMF_F64 ? 0 : 2) + (s.wtype == DMF_W_U16 ? 1 : 0);
    return f[i](a, b, c);
}
kern_t (*g_cost[4])(int, int, int) = {pick_cost_f64_f64, pick_cost_f64_u16, pick_cost_f32_f32, pick_cost_f32_u16};
kern_t (*g_alpha[4])(int, int, int) = {pick_alpha_f64_f64, pick_alpha_f64_u16, pick_alpha_f32_f32, pick_alpha_f32_u16};
kern_t (*g_u[4])(int, int, int) = {pick_u_f64_f64, pick_u_f64_u16, pick_u_f32_f32, pick_u_f32_u16};
kern_t (*g_rowgram[4])(int, int, int) = {pick_rowgram_f64_f64, pick_rowgram_f64_u16, pick_rowgram_f32_f32, pick_rowgram_f32_u16};
kern_t (*g_panel[4])(int, int, int) = {pick_panel_f64_f64, pick_panel_f64_u16, pick_panel_f32_f32, pick_panel_f32_u16};
kern_t (*g_uinner[4])(int, int, int) = {pick_uinner_f64_f64, pick_uinner_f64_u16, pick_uinner_f32_f32, pick_uinner_f32_u16};
kern_t (*g_ainner[4])(int, int, int) = {pick_ainner_f64_f64, pick_ainner_f64_u16, pick_ainner_f32_f32, pick_ainner_f32_u16};
fused_kern_t (*g_fused[4])(int, int, int) = {pick_fused_f64_f64, pick_fused_f64_u16, pick_fused_f32_f32, pick_fused_f32_u16};

fused_kern_t by_types_f(const dmf_shape_t& s, int kb, int nub, int sblk) {
    const int i = (s.dtype == DMF_F64 ? 0 : 2) + (s.wtype == DMF_W_U16 ? 1 : 0);
    return g_fused[i](kb, nub, sblk);
}

// ---------------------------------------------------------------------------------------------
// Geometry.  One stage of the ring holds tile_rows rows of every streamed matrix (X, D, Rk, U, Uprev).
struct StageLayout { size_t off[kMaxSrc], bytes, tx[kMaxSrc]; };
// `row`: bytes per row of each matrix in the stage, `copy`: bytes per row that a tile copies; `x_tail` bytes follow the X rows.
// Every matrix starts 128-byte aligned.
StageLayout stage_layout(long long rows, const size_t (&row)[kMaxSrc], const size_t (&copy)[kMaxSrc], size_t x_tail = 0) {
    StageLayout L{};
    size_t o = 0;
    for (int i = 0; i < kMaxSrc; ++i) {
        L.off[i] = o;
        L.tx[i] = rows * copy[i];
        o = align_up(o + rows * row[i] + (i == 0 ? x_tail : 0), 128);
    }
    L.bytes = o;
    return L;
}
void set_stages(Geom& g, const StageLayout& L) {
    g.offX = (unsigned)L.off[0]; g.offD = (unsigned)L.off[1]; g.offR = (unsigned)L.off[2]; g.offU = (unsigned)L.off[3]; g.offUp = (unsigned)L.off[4];
    g.stage_bytes = (unsigned)L.bytes;
    for (int i = 0; i < kMaxSrc; ++i) g.tile_tx[i] = (unsigned)L.tx[i];
}

// CTAs per fit: fill the GPU (SMs x occupancy) across the whole batch, never more than tiles.  Multi-fit batches: fits terminate
// at different outer iterations, so every fit gets at least 32 CTAs (the grid is oversubscribed, terminated fits return at once)
// and the stragglers still spread over the GPU.
int ctas_per_fit(const dmf_handle_s* h, const dmf_shape_t& s, int occ, int n_tiles) {
    long long per_fit = std::max<long long>(s.n_fits > 1 ? 32 : 1, (long long)h->sm_count * occ / s.n_fits);
    if (s.max_ctas_per_fit > 0) per_fit = std::min<long long>(per_fit, s.max_ctas_per_fit);
    return (int)std::min<long long>(per_fit, n_tiles);
}
int groups_of(int parts) { return (parts + kGroup - 1) / kGroup; }

// Launch geometry of every engine for one shape.  Engines the shape cannot use keep their zero values.
struct Plan {
    // stream engine: cost / alpha / U passes (g.ntc and g.rg are set per launch)
    Geom g;
    int ktb, c_alpha, ntc_alpha;          // alpha / cost kernels: register-row bucket, columns per thread
    int kb, nub, c_u, ntc_u;              // U kernel buckets
    unsigned smem_alpha, smem_u, smem_cost;
    // Gram-form engine (dmf_gram.cuh): own tile geometry, no u_prev in the stage
    int gram_ok;
    Geom gg;
    int kb_g, nub_g, c_g, ntc_g, pb_g, c_p, ntc_p, ktb_in;
    int n_parts_u, n_groups_u;     // u_inner_kernel: one thread per row, many more CTAs than the streaming passes
    unsigned smem_rg, smem_panel;
    int mult_ok;                   // multiplicity form (bootstrap resamples) available for this shape
    unsigned tx_mult[kMaxSrc];     // gg.tile_tx of the multiplicity form: per-source-row sums and multiplicities instead of U, Uprev
    // the 128-register panel variant of the multiplicity form (one unknown type) gets smaller tiles of its own: two CTAs per SM
    int p1_ok;
    Geom gp1;
    unsigned smem_p1;
    // fused engine (dmf_fused.cuh)
    int fused_ok, kb_f, nub_f, s_f;
    FusedShape fc;
    FusedArgs fa;                  // launch template (geometry, stage layout); fits / iteration arguments are filled per launch
    unsigned smem_f;
    // workspace layout
    size_t ws_bytes, off_fits, off_states, off_tickets, off_part, off_gpart, per_fit_tickets, per_fit_part, per_fit_gpart;
    size_t off_usum, per_fit_usum;
    size_t off_rowgram, off_stats, off_gstats, off_red, per_fit_rowgram, per_fit_stats, per_fit_red;
    size_t stats_gbx, stats_scal;      // offsets (in doubles) of gbx and scal inside a per-fit stats block [gram | gbx | scal(8)]
};

int make_plan(const dmf_handle_s* h, const dmf_shape_t& s, Plan& p) {
    p = Plan{};
    if (s.M <= 0 || s.N <= 0 || s.K < 0 || s.n_u <= 0 || s.n_fits <= 0) return fail(DMF_E_SHAPE, "M, N, n_u, n_fits must be positive and K >= 0");
    if (s.mode == DMF_MODE_UNSUPERVISED && s.K != 0) return fail(DMF_E_SHAPE, "unsupervised mode requires K = 0");
    if (s.mode == DMF_MODE_PURITY && s.K == 0) return fail(DMF_E_SHAPE, "purity mode requires K >= 1");
    if (s.dtype != DMF_F64 && s.dtype != DMF_F32) return fail(DMF_E_ARG, "dtype must be DMF_F64 or DMF_F32");
    if (s.wtype != DMF_W_FLOAT && s.wtype != DMF_W_U16) return fail(DMF_E_ARG, "wtype must be DMF_W_FLOAT or DMF_W_U16");
    const int Kp = s.K + (s.K & 1), nup = s.n_u + (s.n_u & 1);
    if (s.ldx < s.N || s.ldd < s.N || s.ldr < Kp || s.ldu < nup) return fail(DMF_E_SHAPE, "row pitch smaller than the (even-padded) row");
    if ((s.ldx | s.ldd | s.ldu | (s.K ? s.ldr : 0)) & 1) return fail(DMF_E_SHAPE, "row pitches must be even (zero padded)");
    const size_t sT = s.dtype == DMF_F64 ? 8 : 4;
    const size_t sW = s.wtype == DMF_W_U16 ? 2 : sT;
    if (s.u_slot < s.M * s.ldu || (s.u_slot * sT) % 16) return fail(DMF_E_SHAPE, "u_slot must be >= M*ldu and a multiple of 16 bytes");
    if (s.u_slots != 0 && s.u_slots != 2 && s.u_slots != 4) return fail(DMF_E_SHAPE, "u_slots must be 2 (or 0) or 4");
    const int Kt = s.K + s.n_u;
    const int rowlen = Kp + nup;
    if (rowlen > kMaxKt || Kt > kMaxKt) return fail(DMF_E_SHAPE, "K + n_u (even padded) > 32 is not supported by this build");
    p.ktb = rowlen <= 8 ? 8 : (rowlen <= 16 ? 16 : 32);
    p.c_alpha = p.ktb <= 16 ? 2 : 1;
    const KernEntry* ue = nullptr;
    for (const KernEntry& e : kUTable)
        if (e.kb >= Kp && e.nub >= nup) { ue = &e; break; }
    if (!ue) return fail(DMF_E_SHAPE, "no U-pass instantiation for this K / n_u");
    p.kb = ue->kb; p.nub = ue->nub; p.c_u = ue->c;
    if (s.N > kConsumers * p.c_alpha || s.N > kConsumers * p.c_u)
        return fail(DMF_E_SHAPE, "N too large for this K + n_u in this build (N <= 512 for small K + n_u, <= 256 otherwise)");
    p.ntc_alpha = pow2ceil((s.N + p.c_alpha - 1) / p.c_alpha);
    p.ntc_u = pow2ceil((s.N + p.c_u - 1) / p.c_u);
    const int rg_u = kConsumers / p.ntc_u;

    const size_t px = s.ldx * sT, pd = s.ldd * sW, pr = s.K ? s.ldr * sT : 0, pu = (size_t)s.ldu * sT;
    // smallest row multiple that keeps every tile start 16-byte aligned
    int ra = 1;
    while (ra < 16 && ((ra * px) % 16 || (ra * pd) % 16 || (ra * pr) % 16 || (ra * pu) % 16)) ra <<= 1;
    const size_t smem_cap = (size_t)h->max_smem_optin;
    const size_t rows_s[kMaxSrc] = {px, pd, pr, pu, pu};
    int occ = std::min(pass_min_blocks(p.ktb), u_pass_min_blocks(p.kb, p.nub, p.c_u));
    int rpt = 0;
    for (int attempt = 0; attempt < 2 && !rpt; ++attempt) {
        const size_t budget = (occ == 2 ? std::min<size_t>(smem_cap, 112 * 1024) : std::min<size_t>(smem_cap, 220 * 1024)) - kCtlBytes - 4096;
        for (int r = ue->rpt; r >= 1; r >>= 1) {
            const long long tr = (long long)r * rg_u;
            if (tr % ra) continue;
            if (stage_layout(tr, rows_s, rows_s).bytes * kStages + (size_t)2 * tr * s.n_u * ((p.ntc_u + 31) / 32) * 8 <= budget) { rpt = r; break; }
        }
        if (!rpt) {
            if (occ == 2) occ = 1; else break;
        }
    }
    if (!rpt) return fail(DMF_E_SHAPE, "one row tile does not fit in shared memory (or pitches force an unsupported tile alignment)");
    const long long tr = (long long)rpt * rg_u;
    Geom& g = p.g;
    g.M = s.M; g.N = s.N; g.K = s.K; g.nu = s.n_u; g.Kt = Kt;
    g.ldx = s.ldx; g.ldd = s.ldd; g.ldr = s.K ? s.ldr : 0; g.ldu = s.ldu;
    g.Kp = Kp; g.nup = nup; g.rpt = rpt;
    g.uslot_bytes = s.u_slot * sT;
    g.tile_rows = (int)tr;
    g.n_tiles = (int)((s.M + tr - 1) / tr);
    g.ntc = p.ntc_alpha; g.rg = kConsumers / p.ntc_alpha;
    g.n_parts = ctas_per_fit(h, s, occ, g.n_tiles);
    g.n_groups = groups_of(g.n_parts);
    set_stages(g, stage_layout(tr, rows_s, rows_s));
    g.row_bulk = (px % 16 == 0 ? 1u : 0u) | (pd % 16 == 0 ? 2u : 0u) | ((pr % 16 == 0 && pr) ? 4u : 0u);
    g.mode = s.mode;
    g.stages = kStages;
    int part_stride = (int)align_up((size_t)std::max(Kt * s.N, 4), 2);

    const size_t pipe = kCtlBytes + (size_t)kStages * g.stage_bytes;
    const size_t epi_alpha = kCtlBytes + ((size_t)(Kt + 1) * s.N + 32) * 8;
    const int wpr_u = (p.ntc_u + 31) / 32;
    const size_t red_u = wpr_u > 1 ? (size_t)2 * tr * wpr_u * s.n_u * 8 : 0;
    p.smem_alpha = (unsigned)std::max(pipe, epi_alpha);
    p.smem_u = (unsigned)std::max(pipe + red_u, (size_t)kCtlBytes + 512);
    p.smem_cost = (unsigned)std::max(pipe, (size_t)kCtlBytes + 512);
    if (std::max(p.smem_alpha, p.smem_u) > smem_cap) return fail(DMF_E_SHAPE, "shared-memory plan exceeds the device limit");

    // ---- Gram-form engine (dmf_gram.cuh): the first kRowgramTable entry that covers K and n_u (n_u <= 4, or n_u <= 8 when K <= 6)
    const KernEntry* ge = nullptr;
    for (const KernEntry& e : kRowgramTable)
        if (e.kb >= Kp && e.nub >= s.n_u) { ge = &e; break; }
    if (ge) {
        p.kb_g = ge->kb; p.nub_g = ge->nub; p.c_g = ge->c;
        // rows per thread and tile: the 4-column kernels walk a tile in batches of their register rows, 4 rows per thread and tile for all
        const int rpt_g_max = p.c_g == 4 ? 4 : ge->rpt;
        const int ng = ng_of(p.nub_g);
        p.pb_g = rowlen <= 8 ? 8 : 16;
        p.c_p = p.pb_g == 8 ? 4 : 1;
        p.ktb_in = Kt <= 8 ? 8 : (Kt <= 16 ? 16 : 32);
        if (s.N <= kConsumers * p.c_g && s.N <= kConsumers * p.c_p) {
            p.ntc_g = pow2ceil((s.N + p.c_g - 1) / p.c_g);
            p.ntc_p = pow2ceil((s.N + p.c_p - 1) / p.c_p);
            const int wpr_g = (p.ntc_g + 31) / 32;
            const int rg_g = kConsumers / p.ntc_g;
            int occ_g = std::min(rowgram_min_blocks(p.kb_g, p.nub_g, p.c_g, rpt_g_max), panel_min_blocks(2, p.pb_g, p.c_p));
            // the U region also holds the per-source-row sums of the multiplicity form (NG doubles per row), followed by the multiplicities
            const size_t rows_g[kMaxSrc] = {px, pd, pr, std::max(pu, (size_t)ng * 8), 4};
            const size_t copy_g[kMaxSrc] = {px, pd, pr, pu, 0}, copy_m[kMaxSrc] = {px, pd, pr, (size_t)ng * 8, 4};
            const size_t epi_panel = kCtlBytes + (size_t)(p.pb_g + 1) * s.N * 8 + 256;
            int rpt_g = 0, stages_g = kStages;
            for (int attempt = 0; attempt < 2 && !rpt_g; ++attempt) {
                const size_t budget = (occ_g == 2 ? std::min<size_t>(smem_cap, 112 * 1024) : std::min<size_t>(smem_cap, 220 * 1024)) - kCtlBytes - 1024;
                // full rows-per-thread first (register slots beyond rpt would be dead work), with a shallower ring if need be
                for (int r = rpt_g_max; r >= 1 && !rpt_g; r = (p.c_g == 4 ? r >> 1 : r - 1)) {
                    const long long trg = (long long)r * rg_g;
                    if (trg % ra) continue;
                    for (int stg = kStages; stg >= 3; --stg)
                        if (stage_layout(trg, rows_g, copy_g).bytes * stg <= budget && epi_panel <= budget + kCtlBytes) { rpt_g = r; stages_g = stg; break; }
                }
                if (!rpt_g) {
                    if (occ_g == 2) occ_g = 1; else break;
                }
            }
            if (rpt_g) {
                const long long trg = (long long)rpt_g * rg_g;
                Geom& q = p.gg;
                q = g;
                q.rpt = rpt_g;
                q.tile_rows = (int)trg; q.n_tiles = (int)((s.M + trg - 1) / trg);
                q.ntc = p.ntc_g; q.rg = rg_g;
                q.n_parts = ctas_per_fit(h, s, occ_g, q.n_tiles);
                q.n_groups = groups_of(q.n_parts);
                q.stages = stages_g;
                set_stages(q, stage_layout(trg, rows_g, copy_g));
                const StageLayout lm = stage_layout(trg, rows_g, copy_m);
                for (int i = 0; i < kMaxSrc; ++i) p.tx_mult[i] = (unsigned)lm.tx[i];
                p.mult_ok = (p.c_g == 4 && p.pb_g == 8 && p.nub_g <= 4 && trg % 4 == 0 && s.mode != DMF_MODE_UNSUPERVISED) ? 1 : 0;
                p.per_fit_usum = p.mult_ok ? align_up((size_t)s.M * ng * 8, 256) : 0;
                if (p.mult_ok && s.n_u == 1) {
                    const size_t budget1 = std::min<size_t>(smem_cap, 112 * 1024) - kCtlBytes - 1024;
                    for (long long tr1 = trg / 2; tr1 >= 4 && !p.p1_ok; tr1 /= 2) {
                        if (tr1 % ra || tr1 % 4) continue;
                        const StageLayout l1 = stage_layout(tr1, rows_g, copy_m);
                        for (int stg = kStages; stg >= 3; --stg)
                            if (l1.bytes * stg <= budget1 && epi_panel <= budget1 + kCtlBytes) {
                                Geom& r = p.gp1;
                                r = q;
                                r.tile_rows = (int)tr1; r.n_tiles = (int)((s.M + tr1 - 1) / tr1); r.stages = stg;
                                r.rpt = 1;                                  // unused by the panel kernel (it strides over the rows of a tile)
                                r.n_parts = std::min(q.n_parts, r.n_tiles); r.n_groups = groups_of(r.n_parts);
                                set_stages(r, l1);
                                p.smem_p1 = (unsigned)std::max(kCtlBytes + (size_t)stg * r.stage_bytes, epi_panel);
                                p.p1_ok = 1;
                                break;
                            }
                    }
                }
                p.n_parts_u = (int)std::min<long long>((s.M + kThreads - 1) / kThreads, std::max<long long>(q.n_parts, (long long)h->sm_count * 8 / s.n_fits));
                p.n_groups_u = groups_of(p.n_parts_u);
                const size_t pipe_g = kCtlBytes + (size_t)stages_g * q.stage_bytes;
                p.smem_rg = (unsigned)std::max(pipe_g, (size_t)kCtlBytes + 512);
                p.smem_panel = (unsigned)std::max(pipe_g, epi_panel);
                part_stride = std::max(part_stride, (int)align_up((size_t)2 * (p.pb_g + 1) * s.N, 2));
                p.per_fit_rowgram = align_up((size_t)s.M * wpr_g * ng * 8, 256);
                p.stats_gbx = (size_t)Kt * Kt * s.N;
                p.stats_scal = p.stats_gbx + (size_t)Kt * s.N;
                p.per_fit_stats = align_up((p.stats_scal + 8) * 8, 256);
                p.per_fit_red = align_up((size_t)part_stride * 8, 256);
                p.gram_ok = 1;
            }
        }
    }
    // ---- fused engine (dmf_fused.cuh): FP64, n_u <= 2, K <= 8, N <= 256, four U slots, rows that bulk copies can place one by one
    if (p.gram_ok && s.dtype == DMF_F64 && s.n_u <= 2 && s.K <= 8 && s.N <= 256 && s.u_slots >= 4 && (s.ldd * sW) % 16 == 0) {
        p.kb_f = s.K == 0 ? 0 : (s.K <= 4 ? 4 : (s.K <= 6 ? 6 : 8));
        p.nub_f = s.n_u;
        p.s_f = s.N <= 64 ? 1 : (s.N <= 128 ? 2 : 4);
        p.fc = fused_shape(p.s_f, p.nub_f);          // rows per tile, ring depth and statistics buffers of the width class
        const int ng = ng_of(p.nub_f), ncol = p.nub_f * p.kb_f + (ng - p.nub_f);
        // a tile is ONE bulk copy per matrix: it keeps the caller's row pitch in shared memory (dmf_shape_t recommends pitches that
        // are free of bank conflicts); 16 zero bytes behind the X rows of every stage serve the panel columns that do not exist.
        const StageLayout lf = stage_layout(p.fc.rows, rows_s, rows_s, 16);
        FusedArgs& fa = p.fa;
        fa.pitchX = (unsigned)px;
        fa.pitchD = (unsigned)pd;
        fa.zero_off = (unsigned)((size_t)p.fc.rows * px);
        fa.offD = (unsigned)lf.off[1]; fa.offR = (unsigned)lf.off[2]; fa.offU = (unsigned)lf.off[3]; fa.offUp = (unsigned)lf.off[4];
        fa.stage_bytes = (unsigned)lf.bytes;
        fa.offStats = kFusedCtlBytes + p.fc.stages * fa.stage_bytes;
        // row statistics (one partial per A-warp sample group and row; nstat buffers), then the per-sample table of the A-warps
        fa.offTab = (unsigned)align_up(fa.offStats + (unsigned)p.fc.nstat * p.fc.sgroups * p.fc.rows * ng * 8u, 128);
        p.smem_f = fa.offTab + 32u * p.s_f * 2u * p.nub_f * 8u;
        const size_t n_rec = 2 + (size_t)(ncol + p.nub_f) * s.N;
        if (p.smem_f <= smem_cap && kFusedCtlBytes + n_rec * 8 <= fa.offStats) {
            fa.n_tiles = (int)((s.M + p.fc.rows - 1) / p.fc.rows);
            fa.g = g;
            fa.g.n_parts = ctas_per_fit(h, s, 1, fa.n_tiles);
            fa.g.n_groups = groups_of(fa.g.n_parts);
            part_stride = std::max(part_stride, (int)align_up(n_rec, 2));
            p.per_fit_red = align_up((size_t)part_stride * 8, 256);
            p.fused_ok = 1;
        }
    }
    // one partial-record stride for every engine: they share the workspace
    for (Geom* q : {&p.g, &p.gg, &p.gp1, &p.fa.g}) q->part_stride = part_stride;
    const int parts_max = std::max({p.g.n_parts, p.gg.n_parts, p.fa.g.n_parts});
    const int groups_max = std::max({p.g.n_groups, p.gg.n_groups, p.n_groups_u, p.fa.g.n_groups});
    // u_inner_kernel records are 8 doubles apart: n_parts_u * 8 <= parts_max * part_stride holds because part_stride >= 2 * 9 * N

    // workspace layout
    p.off_fits = 0;
    p.off_states = align_up(p.off_fits + sizeof(FitDev) * s.n_fits, 256);
    p.per_fit_tickets = align_up(sizeof(unsigned) * (groups_max + 1), 128);
    p.per_fit_part = align_up((size_t)parts_max * part_stride * 8, 128);
    p.per_fit_gpart = align_up((size_t)groups_max * part_stride * 8, 128);
    p.off_tickets = align_up(p.off_states + sizeof(FitState) * s.n_fits, 256);
    p.off_part = align_up(p.off_tickets + p.per_fit_tickets * s.n_fits, 256);
    p.off_gpart = align_up(p.off_part + p.per_fit_part * s.n_fits, 256);
    p.off_rowgram = align_up(p.off_gpart + p.per_fit_gpart * s.n_fits, 256);
    p.off_stats = p.off_rowgram + p.per_fit_rowgram * s.n_fits;       // this GPU's statistics, fits contiguous
    p.off_gstats = p.off_stats + p.per_fit_stats * s.n_fits;          // all-reduced copies (row-sharded runs)
    p.off_red = p.off_gstats + p.per_fit_stats * s.n_fits;
    p.off_usum = p.off_red + p.per_fit_red * s.n_fits;
    p.ws_bytes = align_up(p.off_usum + p.per_fit_usum * s.n_fits, 256);
    return DMF_OK;
}

}  // namespace

struct dmf_batch_s {
    dmf_handle_s* h;
    dmf_shape_t shape;
    Plan p;                 // make_plan, adjusted to the batch by dmf_batch_create (gather, multiplicity form, engines it rules out)
    FitDev* fits_dev;       // in workspace
    FitState* states_dev;   // in workspace, contiguous [n_fits]
    long long launches;
    FitState* pinned;       // host staging for state polling
    int engine;             // DMF_ENGINE_*
    int n_active;                   // fits_dev holds the descriptors of the first n_active still-running fits (compacted at every poll)
    // peer exchange (row-sharded runs): symmetric buffers of all ranks, see peer_allreduce_kernel
    double** peers_dev;             // device array [world]
    unsigned* xchg_ticket;          // device
    int peer_rank, peer_world;
    long long peer_slot_stride, peer_flag_off;
    unsigned xchg_epoch;
    int fused_pending;              // a dmf_fused_outer ran since the cost of the current iterate was last evaluated
    int multmode;                   // fits are bootstrap resamples in multiplicity form
    int sharded;                    // CpG rows sharded over GPUs: kernels publish partial sums, finalize runs on all-reduced sums
    std::vector<FitDev> fits_host;
    double *stats_local, *stats_global;
    // momentum table (library-owned, grows on demand): a_t and (a_t - 1) / a_{t+1}
    std::vector<double> mom_host;   // [a_0 .. a_{n-1} | m_0 .. m_{n-1}] is rebuilt on growth
    double* mom_dev;
    size_t mom_cap;                 // entries per array on the device
    long long t_hi;                 // upper bound of the inner-iteration index any fit of the batch can have reached
};

namespace {

// Make sure the device momentum table covers indices [0, need].  Growth synchronises the stream (rare: the table doubles).
int ensure_mom(dmf_batch_s* b, long long need, cudaStream_t st) {
    if ((size_t)need + 1 <= b->mom_cap) return DMF_OK;
    size_t cap = std::max<size_t>(4096, b->mom_cap * 2);
    while (cap < (size_t)need + 1) cap *= 2;
    std::vector<double> h(2 * cap);
    volatile double a0 = 1.0;
    for (size_t t = 0; t < cap; ++t) {
        volatile double sq = 4.0 * a0;
        sq = sq * a0;
        sq = 1.0 + sq;
        volatile double a1 = (1.0 + sqrt((double)sq)) / 2.0;     // deconvolution.py:84, same operation order as the device code
        h[t] = a0;
        h[cap + t] = (a0 - 1.0) / a1;
        a0 = a1;
    }
    double* dev = nullptr;
    CUDA_TRY(cudaMalloc(&dev, 2 * cap * sizeof(double)));
    cudaError_t e = cudaMemcpyAsync(dev, h.data(), 2 * cap * sizeof(double), cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);      // also retires every launch that still reads the old table
    if (e != cudaSuccess) {
        cudaFree(dev);
        return fail(DMF_E_CUDA, std::string("momentum table: ") + cudaGetErrorString(e));
    }
    if (b->mom_dev) cudaFree(b->mom_dev);
    b->mom_dev = dev;
    b->mom_cap = cap;
    return DMF_OK;
}

// Upload the descriptors of the fits listed in `ids` (all fits when ids == nullptr) to the front of fits_dev.
int upload_fits(dmf_batch_s* b, const std::vector<int>* ids, cudaStream_t st) {
    const int n = ids ? (int)ids->size() : b->shape.n_fits;
    if (n == 0) { b->n_active = 0; return DMF_OK; }
    std::vector<FitDev> tmp;
    const FitDev* src = b->fits_host.data();
    if (ids) {
        tmp.resize(n);
        for (int i = 0; i < n; ++i) tmp[i] = b->fits_host[(*ids)[i]];
        src = tmp.data();
    }
    CUDA_TRY(cudaMemcpyAsync(b->fits_dev, src, sizeof(FitDev) * n, cudaMemcpyHostToDevice, st));   // pageable source: staged before return
    b->n_active = n;
    return DMF_OK;
}

int set_smem(kern_t k, unsigned bytes) {
    if (!k) return fail(DMF_E_SHAPE, "no kernel instantiation for this shape");
    CUDA_TRY(cudaFuncSetAttribute((const void*)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes));
    return DMF_OK;
}

int launch(dmf_batch_s* b, kern_t k, int ntc, unsigned smem, int flags, int k_inner, double tol, cudaStream_t st) {
    if (!k) return fail(DMF_E_SHAPE, "no kernel instantiation for this shape");
    if (b->multmode) return fail(DMF_E_STATE, "fits in multiplicity form run on the Gram-form engine only (dmf_gram_*)");
    PassArgs a;
    a.g = b->p.g;
    a.g.ntc = ntc;
    a.g.rg = kConsumers / ntc;
    a.fits = b->fits_dev;
    a.k_inner = k_inner;
    a.flags = flags;
    a.tol = tol;
    a.ca0 = a.cb0 = a.with_x = a.pad = 0;
    a.mom_a = b->mom_dev; a.mom_m = b->mom_dev ? b->mom_dev + b->mom_cap : nullptr;
    dim3 grid(a.g.n_parts, b->n_active, 1);
    k<<<grid, kThreads, smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    b->launches++;
    return DMF_OK;
}

kern_t k_cost(dmf_batch_s* b, int initial) { return by_types(b->shape, g_cost, b->p.ktb, initial, b->p.c_alpha); }
kern_t k_alpha(dmf_batch_s* b) { return by_types(b->shape, g_alpha, b->p.ktb, 0, b->p.c_alpha); }
kern_t k_u(dmf_batch_s* b) { return by_types(b->shape, g_u, b->p.kb, b->p.nub, 0); }
kern_t k_rowgram(dmf_batch_s* b, int initial) { return by_types(b->shape, g_rowgram, b->p.kb_g, b->p.nub_g, initial); }
kern_t k_panel(dmf_batch_s* b) { return by_types(b->shape, g_panel, b->p.pb_g, b->p.c_p, b->multmode); }
kern_t k_panel_u1(dmf_batch_s* b) { return by_types(b->shape, g_panel, b->p.pb_g, b->p.c_p, 2); }     // multiplicity form, n_u == 1
kern_t k_uinner(dmf_batch_s* b) { return by_types(b->shape, g_uinner, b->p.nub_g, b->multmode ? 1 : 0, 0); }
kern_t k_costcross(dmf_batch_s* b) { return by_types(b->shape, g_uinner, b->p.nub_g, 2, 0); }
kern_t k_usum(dmf_batch_s* b) { return by_types(b->shape, g_uinner, b->p.nub_g, 3, 0); }
kern_t k_ainner(dmf_batch_s* b) { return by_types(b->shape, g_ainner, b->p.ktb_in, 0, 0); }

// Gram-engine launch: geometry gg; ntc selects the thread mapping of the kernel; grid_x CTAs per fit (0: one CTA per fit on grid.x)
int launch_g(dmf_batch_s* b, kern_t k, int ntc, unsigned smem, int flags, int k_inner, double tol, int ca0, int cb0, int with_x,
             int grid_mode /* 0: pass grid, 1: one CTA per fit, 2: wide row grid of u_inner_kernel */, cudaStream_t st,
             const Geom* geom = nullptr) {
    if (!k) return fail(DMF_E_SHAPE, "no Gram-engine kernel instantiation for this shape");
    PassArgs a;
    a.g = geom ? *geom : b->p.gg;
    a.g.ntc = ntc;
    a.g.rg = kConsumers / ntc;
    a.fits = b->fits_dev;
    a.k_inner = k_inner;
    a.flags = flags | (b->sharded ? kFlagPartial : 0);
    a.tol = tol;
    a.ca0 = ca0; a.cb0 = cb0; a.with_x = with_x; a.pad = 0;
    a.mom_a = b->mom_dev; a.mom_m = b->mom_dev + b->mom_cap;
    // grid_mode 1 (alpha_inner_kernel): one warp per 32 / L samples of a fit, L = ktb_in lanes per sample
    const int spw = 32 / b->p.ktb_in;
    dim3 grid = grid_mode == 1 ? dim3(b->n_active, (b->shape.N + spw - 1) / spw, 1) : dim3(a.g.n_parts, b->n_active, 1);
    if (grid_mode == 2) {
        a.g.n_parts = b->p.n_parts_u;
        a.g.n_groups = b->p.n_groups_u;
        if (b->p.n_parts_u != b->p.gg.n_parts) a.g.part_stride = 8;
        grid = dim3(b->p.n_parts_u, b->n_active, 1);
    }
    if (grid_mode == 1) a.g.fit_major = 0;
    else if (a.g.fit_major) {
        if (grid.x > 65535u) a.g.fit_major = 0;          // grid.y limit
        else grid = dim3(grid.y, grid.x, 1);
    }
    k<<<grid, grid_mode == 1 ? 32 : kThreads, smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    b->launches++;
    return DMF_OK;
}

// ---------------------------------------------------------------------------------------------
// small utility kernels
template <typename S>
__global__ void pack_u16_kernel(const S* src, long long n, uint16_t* dst, int* bad) {
    int local_bad = 0;
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const S v = src[i];
        const double d = (double)v;
        const bool ok = d >= 0.0 && d <= 65535.0 && d == floor(d);
        if (!ok) local_bad = 1;
        dst[i] = ok ? (uint16_t)d : (uint16_t)0;
    }
    if (local_bad) atomicAdd(bad, 1);
}

__global__ void gather_rows_kernel(const char* src, const int32_t* rows, long long n_rows, long long row_bytes, char* dst) {
    // one warp per destination row; 16-byte vectors when the row allows it
    const long long warp = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = warp; r < n_rows; r += nwarps) {
        const char* s = src + (long long)rows[r] * row_bytes;
        char* d = dst + r * row_bytes;
        if ((row_bytes & 15) == 0 && ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0) {
            for (long long o = lane * 16LL; o < row_bytes; o += 512) *reinterpret_cast<int4*>(d + o) = *reinterpret_cast<const int4*>(s + o);
        } else {
            for (long long o = lane; o < row_bytes; o += 32) d[o] = s[o];
        }
    }
}

// dmf_batch_set_step_state: the scalars of up to kStepChunk fits travel in the kernel parameters, so the call needs no device
// staging buffer and returns without waiting for the stream
constexpr int kStepChunk = 128;
struct StepStateArgs {
    FitState* st;
    int which, n;
    double a[kStepChunk], l[kStepChunk], l_old[kStepChunk];
};

__global__ void set_step_state_kernel(const StepStateArgs s) {
    const int i = threadIdx.x;
    if (i >= s.n) return;
    FitState& f = s.st[i];
    if (s.which == 0) { f.a1 = s.a[i]; f.l_w = s.l[i]; f.l_w_old = s.l_old[i]; }
    else { f.a2 = s.a[i]; f.l_h = s.l[i]; f.l_h_old = s.l_old[i]; }
}

}  // namespace

// =================================================================================================
extern "C" {

int dmf_abi_version(void) { return DMF_ABI_VERSION; }
const char* dmf_last_error(void) { return g_err.c_str(); }

int dmf_create(int device, dmf_handle_t* out) {
    if (!out) return fail(DMF_E_ARG, "out is NULL");
    int n = 0;
    CUDA_TRY(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(DMF_E_ARG, "no such CUDA device");
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(DMF_E_CUDA, "libdemethify_sm100 requires an sm_100-class (Blackwell) GPU");
    dmf_handle_s* h = new dmf_handle_s;
    h->device = device;
    h->sm_count = prop.multiProcessorCount;
    h->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    *out = h;
    return DMF_OK;
}

int dmf_destroy(dmf_handle_t h) {
    delete h;
    return DMF_OK;
}

int dmf_sm_count(dmf_handle_t h, int* out) {
    if (!h || !out) return fail(DMF_E_ARG, "NULL argument");
    *out = h->sm_count;
    return DMF_OK;
}

int dmf_batch_workspace_bytes(dmf_handle_t h, const dmf_shape_t* shape, size_t* bytes) {
    if (!h || !shape || !bytes) return fail(DMF_E_ARG, "NULL argument");
    Plan p;
    int rc = make_plan(h, *shape, p);
    if (rc) return rc;
    *bytes = p.ws_bytes;
    return DMF_OK;
}

int dmf_batch_create(dmf_handle_t h, const dmf_shape_t* shape, const dmf_fit_desc_t* fits, void* ws, size_t ws_bytes,
                     void* stream, dmf_batch_t* out) {
    if (!h || !shape || !fits || !ws || !out) return fail(DMF_E_ARG, "NULL argument");
    Plan p;
    int rc = make_plan(h, *shape, p);
    if (rc) return rc;
    if (ws_bytes < p.ws_bytes) return fail(DMF_E_ARG, "workspace too small");
    if (reinterpret_cast<uintptr_t>(ws) & 255) return fail(DMF_E_ARG, "workspace must be 256-byte aligned");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    const dmf_shape_t& s = *shape;
    std::vector<FitDev> host(s.n_fits);
    char* base = static_cast<char*>(ws);
    if (p.gram_ok && cudaMemsetAsync(base + p.off_stats, 0, 2 * p.per_fit_stats * s.n_fits, (cudaStream_t)stream) != cudaSuccess)
        return fail(DMF_E_CUDA, "batch set-up: clearing the statistics buffers failed");
    bool gather = false;
    int n_mult = 0;
    bool shared_inputs = s.n_fits > 1;
    for (int i = 0; i < s.n_fits; ++i) {
        const dmf_fit_desc_t& d = fits[i];
        if ((d.mult != nullptr) != (d.offs != nullptr)) return fail(DMF_E_ARG, "fit descriptor: mult and offs go together");
        if (d.mult && !d.rows) return fail(DMF_E_ARG, "fit descriptor: the multiplicity form needs rows (source row of every position, sorted)");
        if (d.mult && (reinterpret_cast<uintptr_t>(d.mult) & 15)) return fail(DMF_E_ARG, "fit descriptor: mult must be 16-byte aligned (it is streamed with bulk copies)");
        n_mult += d.mult ? 1 : 0;
        shared_inputs &= (d.X == fits[0].X && d.D == fits[0].D && d.Rk == fits[0].Rk);
        if (!d.X || !d.D || !d.U || !d.A || (s.K && !d.Rk)) return fail(DMF_E_ARG, "fit descriptor has a NULL matrix");
        if (s.mode == DMF_MODE_PURITY && !d.purity) return fail(DMF_E_ARG, "purity mode needs a purity vector");
        const uintptr_t al = reinterpret_cast<uintptr_t>(d.X) | reinterpret_cast<uintptr_t>(d.D) | reinterpret_cast<uintptr_t>(d.Rk) |
                             reinterpret_cast<uintptr_t>(d.U) | reinterpret_cast<uintptr_t>(d.A);
        if (al & 15) return fail(DMF_E_ARG, "matrix base pointers must be 16-byte aligned");
        FitDev& f = host[i];
        f.X = static_cast<const char*>(d.X);
        f.D = static_cast<const char*>(d.D);
        f.Rk = static_cast<const char*>(d.Rk);
        f.rows = d.mult ? nullptr : d.rows;          // multiplicity form: rows is the position -> source row map, nothing is gathered
        f.pos_row = d.mult ? d.rows : nullptr;
        gather |= (d.rows != nullptr && d.mult == nullptr);
        f.U = static_cast<char*>(d.U);
        f.A = static_cast<char*>(d.A);
        f.purity = d.purity;
        f.trace = d.cost_trace;
        f.trace_cap = d.cost_trace ? d.trace_cap : 0;
        f.part = reinterpret_cast<double*>(base + p.off_part + p.per_fit_part * i);
        f.gpart = reinterpret_cast<double*>(base + p.off_gpart + p.per_fit_gpart * i);
        f.tickets = reinterpret_cast<unsigned*>(base + p.off_tickets + p.per_fit_tickets * i);
        f.st = reinterpret_cast<FitState*>(base + p.off_states) + i;
        f.rowgram = p.gram_ok ? reinterpret_cast<double*>(base + p.off_rowgram + p.per_fit_rowgram * i) : nullptr;
        f.gram = p.gram_ok ? reinterpret_cast<double*>(base + p.off_stats + p.per_fit_stats * i) : nullptr;
        f.gbx = p.gram_ok ? f.gram + p.stats_gbx : nullptr;
        f.scal = p.gram_ok ? f.gram + p.stats_scal : nullptr;
        f.rgram = f.gram; f.rgbx = f.gbx; f.rscal = f.scal;
        f.red = p.gram_ok ? reinterpret_cast<double*>(base + p.off_red + p.per_fit_red * i) : nullptr;
        f.mult = d.mult; f.offs = d.offs;
        f.usum = p.mult_ok ? reinterpret_cast<double*>(base + p.off_usum + p.per_fit_usum * i) : nullptr;
        f.pad = 0;
    }
    if (n_mult && n_mult != s.n_fits) return fail(DMF_E_ARG, "either all fits of a batch are in multiplicity form or none");
    if (n_mult && !p.mult_ok)
        return fail(DMF_E_SHAPE, "the multiplicity form needs K <= 6, n_u <= 4, K + n_u (even padded) <= 8, partial or purity mode and a tile of a multiple of 4 rows");
    dmf_batch_s* b = new dmf_batch_s;
    b->h = h;
    b->shape = s;
    b->p = p;
    b->multmode = n_mult ? 1 : 0;
    b->launches = 0;
    b->pinned = nullptr;
    b->mom_dev = nullptr;
    b->mom_cap = 0;
    b->t_hi = 0;
    b->sharded = 0;
    b->peers_dev = nullptr; b->xchg_ticket = nullptr; b->peer_rank = 0; b->peer_world = 0; b->xchg_epoch = 0;
    b->n_active = s.n_fits;
    b->fits_host = host;
    b->stats_local = p.gram_ok ? reinterpret_cast<double*>(base + p.off_stats) : nullptr;
    b->stats_global = p.gram_ok ? reinterpret_cast<double*>(base + p.off_gstats) : nullptr;
    b->fits_dev = reinterpret_cast<FitDev*>(base + p.off_fits);
    b->states_dev = reinterpret_cast<FitState*>(base + p.off_states);
    b->fused_pending = 0;
    // what the plan leaves to the fits of the batch
    Plan& bp = b->p;
    for (Geom* q : {&bp.g, &bp.gg, &bp.gp1}) q->gather = gather ? 1 : 0;
    bp.gg.multmode = bp.gp1.multmode = b->multmode;
    bp.gg.fit_major = bp.gp1.fit_major = shared_inputs ? 1 : 0;
    if (b->multmode) std::copy(bp.tx_mult, bp.tx_mult + kMaxSrc, bp.gg.tile_tx);
    bp.p1_ok = b->multmode && p.p1_ok;
    bp.fused_ok = p.fused_ok && !gather && !n_mult;
    b->engine = p.gram_ok ? DMF_ENGINE_GRAM : DMF_ENGINE_STREAM;      // multiplicity form implies gram (checked above)
    if (bp.fused_ok) {
        fused_kern_t kf = by_types_f(s, p.kb_f, p.nub_f, p.s_f);
        if (!kf || cudaFuncSetAttribute((const void*)kf, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem_f) != cudaSuccess) {
            cudaGetLastError();
            bp.fused_ok = 0;
        } else {
            b->engine = DMF_ENGINE_FUSED;
        }
    }
    if (p.gram_ok) {
        if ((long long)p.n_parts_u * 8 > (long long)std::max(p.g.n_parts, p.gg.n_parts) * p.g.part_stride ||
            (long long)p.n_groups_u * 8 > (long long)std::max(p.g.n_groups, p.gg.n_groups) * p.g.part_stride) {
            bp.n_parts_u = p.gg.n_parts; bp.n_groups_u = p.gg.n_groups;     // partial-sum buffers too small for the wide grid (tiny N): use the pass grid
        }
        if ((rc = set_smem(k_rowgram(b, 0), p.smem_rg)) || (rc = set_smem(k_rowgram(b, 1), p.smem_rg)) || (rc = set_smem(k_panel(b), p.smem_panel)) ||
            (rc = set_smem(k_uinner(b), 0)) || (rc = set_smem(k_ainner(b), 0)) || (b->multmode && ((rc = set_smem(k_costcross(b), 0)) || (rc = set_smem(k_panel_u1(b), std::max(p.smem_panel, bp.p1_ok ? p.smem_p1 : 0u)))))) {
            delete b;
            return rc;
        }
    }
    if ((rc = set_smem(k_cost(b, 0), p.smem_cost)) || (rc = set_smem(k_cost(b, 1), p.smem_cost)) || (rc = set_smem(k_alpha(b), p.smem_alpha)) ||
        (rc = set_smem(k_u(b), p.smem_u))) {
        delete b;
        return rc;
    }
    // zero states + tickets, upload descriptors (pageable source: the copy is staged before return)
    cudaError_t e = cudaMemsetAsync(base + p.off_states, 0, p.off_part - p.off_states, st);
    if (e == cudaSuccess) e = cudaMemcpyAsync(b->fits_dev, host.data(), sizeof(FitDev) * s.n_fits, cudaMemcpyHostToDevice, st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e == cudaSuccess) e = cudaMallocHost(&b->pinned, sizeof(FitState) * s.n_fits);
    if (e != cudaSuccess) {
        delete b;
        return fail(DMF_E_CUDA, std::string("batch set-up: ") + cudaGetErrorString(e));
    }
    *out = b;
    return DMF_OK;
}

int dmf_batch_destroy(dmf_batch_t b) {
    if (!b) return DMF_OK;
    if (b->pinned) cudaFreeHost(b->pinned);
    if (b->mom_dev) cudaFree(b->mom_dev);
    if (b->peers_dev) cudaFree(b->peers_dev);
    if (b->xchg_ticket) cudaFree(b->xchg_ticket);
    delete b;
    return DMF_OK;
}

int dmf_batch_geometry(dmf_batch_t b, int32_t* ctas_per_fit, int32_t* tile_rows, int32_t* smem_bytes) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    const Plan& p = b->p;
    if (b->engine == DMF_ENGINE_FUSED) {
        if (ctas_per_fit) *ctas_per_fit = p.fa.g.n_parts;
        if (tile_rows) *tile_rows = p.fc.rows;
        if (smem_bytes) *smem_bytes = (int32_t)p.smem_f;
        return DMF_OK;
    }
    if (ctas_per_fit) *ctas_per_fit = b->engine == DMF_ENGINE_GRAM ? p.gg.n_parts : p.g.n_parts;
    if (tile_rows) *tile_rows = b->engine == DMF_ENGINE_GRAM ? p.gg.tile_rows : p.g.tile_rows;
    if (smem_bytes) *smem_bytes = b->engine == DMF_ENGINE_GRAM ? (int32_t)std::max(p.smem_rg, p.smem_panel) : (int32_t)std::max(p.smem_alpha, p.smem_u);
    return DMF_OK;
}

int dmf_pass_init(dmf_batch_t b, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    b->t_hi = 0;
    if (b->n_active != b->shape.n_fits) { int rc0 = upload_fits(b, nullptr, (cudaStream_t)stream); if (rc0) return rc0; }
    return launch(b, k_cost(b, 1), b->p.ntc_alpha, b->p.smem_cost, kFlagInitial, 0, 0.0, (cudaStream_t)stream);
}
int dmf_pass_cost(dmf_batch_t b, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    return launch(b, k_cost(b, 0), b->p.ntc_alpha, b->p.smem_cost, 0, 0, tol, (cudaStream_t)stream);
}
int dmf_pass_u(dmf_batch_t b, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    b->t_hi += 1;     // keeps the momentum-table bound valid if Gram-engine steps follow on the same batch
    return launch(b, k_u(b), b->p.ntc_u, b->p.smem_u, 0, 0, 0.0, (cudaStream_t)stream);
}
int dmf_pass_alpha(dmf_batch_t b, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (b->shape.mode == DMF_MODE_PURITY) return fail(DMF_E_STATE, "purity batches use dmf_pass_fw");
    return launch(b, k_alpha(b), b->p.ntc_alpha, b->p.smem_alpha, 0, 0, 0.0, (cudaStream_t)stream);
}
int dmf_pass_fw(dmf_batch_t b, int32_t k_inner, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (b->shape.mode != DMF_MODE_PURITY) return fail(DMF_E_STATE, "Frank-Wolfe steps need a purity batch");
    return launch(b, k_alpha(b), b->p.ntc_alpha, b->p.smem_alpha, kFlagFW, k_inner, 0.0, (cudaStream_t)stream);
}
int dmf_batch_set_step_state(dmf_batch_t b, int32_t which, const double* a, const double* l, const double* l_old, void* stream) {
    if (!b || !a || !l || !l_old) return fail(DMF_E_ARG, "NULL argument");
    if (which != 0 && which != 1) return fail(DMF_E_ARG, "which must be 0 (a1, l_w, l_w_old) or 1 (a2, l_h, l_h_old)");
    const int n = b->shape.n_fits;
    for (int i = 0; i < n; ++i) {        // every fit is checked before any state is written
        if (!std::isfinite(a[i]) || !std::isfinite(l[i]) || !std::isfinite(l_old[i]))
            return fail(DMF_E_ARG, "step state of fit " + std::to_string(i) + " is not finite");
        if (!(l[i] > 0.0)) return fail(DMF_E_ARG, "step constant l of fit " + std::to_string(i) + " must be positive");
    }
    for (int i0 = 0; i0 < n; i0 += kStepChunk) {
        StepStateArgs s;
        s.st = b->states_dev + i0;
        s.which = which;
        s.n = std::min(kStepChunk, n - i0);
        for (int i = 0; i < s.n; ++i) { s.a[i] = a[i0 + i]; s.l[i] = l[i0 + i]; s.l_old[i] = l_old[i0 + i]; }
        set_step_state_kernel<<<1, kStepChunk, 0, (cudaStream_t)stream>>>(s);
        CUDA_TRY(cudaGetLastError());
        b->launches++;
    }
    return DMF_OK;
}

int dmf_batch_set_engine(dmf_batch_t b, int32_t engine) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (engine != DMF_ENGINE_STREAM && engine != DMF_ENGINE_GRAM && engine != DMF_ENGINE_FUSED) return fail(DMF_E_ARG, "engine must be DMF_ENGINE_STREAM, DMF_ENGINE_GRAM or DMF_ENGINE_FUSED");
    if (engine == DMF_ENGINE_FUSED && !b->p.fused_ok)
        return fail(DMF_E_SHAPE, "the fused engine needs FP64 storage, n_u <= 2, K <= 8, N <= 256, four U slots, no row gather and a weight pitch of a multiple of 16 bytes");
    if (b->fused_pending) return fail(DMF_E_STATE, "the cost of the current iterate is pending (dmf_fused_finish) - engines can be switched after it");
    if (engine == DMF_ENGINE_GRAM && !b->p.gram_ok)
        return fail(DMF_E_SHAPE, "the Gram-form engine supports n_u <= 4 (n_u <= 8 when K <= 6) and needs its tile to fit in shared memory");
    if (engine == DMF_ENGINE_STREAM && b->multmode) return fail(DMF_E_STATE, "fits in multiplicity form run on the Gram-form engine only");
    b->engine = engine;
    return DMF_OK;
}
int dmf_batch_get_engine(dmf_batch_t b, int32_t* engine) {
    if (!b || !engine) return fail(DMF_E_ARG, "NULL argument");
    *engine = b->engine;
    return DMF_OK;
}

int dmf_gram_rowgram(dmf_batch_t b, int32_t initial, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "no Gram-engine instantiation for this shape");
    if (initial) {
        b->t_hi = 0;
        b->fused_pending = 0;
        if (b->n_active != b->shape.n_fits) { int rc0 = upload_fits(b, nullptr, (cudaStream_t)stream); if (rc0) return rc0; }
    }
    int rc = launch_g(b, k_rowgram(b, initial ? 1 : 0), b->p.ntc_g, b->p.smem_rg, initial ? kFlagInitial : 0, 0, tol, 0, 0, 0, 0, (cudaStream_t)stream);
    if (rc || !b->multmode) return rc;
    // multiplicity form: the per-position cost terms and the set-up / termination logic
    return launch_g(b, k_costcross(b), b->p.ntc_g, 0, initial ? kFlagInitial : 0, 0, tol, 0, 0, 0, 2, (cudaStream_t)stream);
}
int dmf_gram_u_inner(dmf_batch_t b, int32_t n_iter2, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "no Gram-engine instantiation for this shape");
    if (b->fused_pending) return fail(DMF_E_STATE, "the row statistics are stale after dmf_fused_outer: dmf_fused_finish first");
    if (n_iter2 < 0) return fail(DMF_E_ARG, "negative iteration count");
    b->t_hi += n_iter2;
    int rc = ensure_mom(b, b->t_hi, (cudaStream_t)stream);
    if (rc) return rc;
    rc = launch_g(b, k_uinner(b), b->p.ntc_g, 0, 0, n_iter2, 0.0, 0, 0, 0, 2, (cudaStream_t)stream);
    if (rc || !b->multmode) return rc;
    return launch_g(b, k_usum(b), b->p.ntc_g, 0, 0, 0, 0.0, 0, 0, 0, 2, (cudaStream_t)stream);      // per-source-row sums for the panel pass
}
int dmf_gram_panels(dmf_batch_t b, int32_t known_block, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "no Gram-engine instantiation for this shape");
    const Plan& p = b->p;
    const int nR = p.gg.Kp >> 1, nU = p.gg.nup >> 1, nb = p.pb_g / 2;
    const int ca_lo = known_block ? 0 : nR, ca_hi = known_block ? nR : nR + nU;
    const int cb_hi = known_block ? nR : nR + nU;
    int rc;
    const bool u1 = b->multmode && !known_block && b->shape.n_u == 1;
    const bool own = u1 && p.p1_ok;                    // smaller tiles, two CTAs per SM
    for (int ca = ca_lo; ca < ca_hi; ++ca)
        for (int cb = 0; cb < cb_hi; cb += nb)
            if ((rc = launch_g(b, u1 ? k_panel_u1(b) : k_panel(b), p.ntc_p, own ? p.smem_p1 : p.smem_panel, 0, p.nub_g, 0.0,
                               ca, cb, cb == 0 ? 1 : 0, 0, (cudaStream_t)stream, own ? &p.gp1 : nullptr))) return rc;
    return DMF_OK;
}
int dmf_gram_alpha_inner(dmf_batch_t b, int32_t n_iter2, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "no Gram-engine instantiation for this shape");
    if (n_iter2 < 0) return fail(DMF_E_ARG, "negative iteration count");
    // alpha steps never run ahead of the U steps by more than one call; cover t_hi + n_iter2 to be independent of call order
    int rc = ensure_mom(b, b->t_hi + n_iter2, (cudaStream_t)stream);
    if (rc) return rc;
    return launch_g(b, k_ainner(b), b->p.ntc_p, 0, b->shape.mode == DMF_MODE_PURITY ? kFlagFW : 0, n_iter2, 0.0, 0, 0, 0, 1, (cudaStream_t)stream);
}
int dmf_batch_set_sharded(dmf_batch_t b, int32_t on, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "row sharding needs the Gram-form engine (n_u <= 4, or n_u <= 8 with K <= 6)");
    if (b->multmode) return fail(DMF_E_STATE, "row sharding and the multiplicity form are not combined");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t per = b->p.per_fit_stats / 8;
    for (int i = 0; i < b->shape.n_fits; ++i) {
        FitDev& f = b->fits_host[i];
        double* src = on ? b->stats_global + per * i : b->stats_local + per * i;
        f.rgram = src; f.rgbx = src + b->p.stats_gbx; f.rscal = src + b->p.stats_scal;
    }
    int rc = upload_fits(b, nullptr, st);
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(st));
    b->sharded = on ? 1 : 0;
    b->engine = b->p.fused_ok ? DMF_ENGINE_FUSED : DMF_ENGINE_GRAM;
    return DMF_OK;
}
int dmf_batch_stats_buffers(dmf_batch_t b, void** local_dev, void** global_dev, int64_t* doubles_per_fit, int64_t* scal_offset) {
    if (!b || !local_dev || !global_dev || !doubles_per_fit || !scal_offset) return fail(DMF_E_ARG, "NULL argument");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "no Gram-engine instantiation for this shape");
    *local_dev = b->stats_local; *global_dev = b->stats_global;
    *doubles_per_fit = (int64_t)(b->p.per_fit_stats / 8); *scal_offset = (int64_t)b->p.stats_scal;
    return DMF_OK;
}
int dmf_gram_finalize_cost(dmf_batch_t b, int32_t initial, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->sharded) return fail(DMF_E_STATE, "dmf_gram_finalize_cost is the second half of dmf_gram_rowgram on row-sharded batches");
    PassArgs a;
    memset(&a, 0, sizeof(a));
    a.g = b->p.gg;
    a.fits = b->fits_dev;
    a.k_inner = b->n_active;
    a.flags = (initial ? kFlagInitial : 0) | (b->shape.dtype == DMF_F32 ? kFlagF32 : 0);
    a.tol = tol;
    finalize_cost_kernel<<<(b->n_active + 127) / 128, 128, 0, (cudaStream_t)stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    b->launches++;
    return DMF_OK;
}

int dmf_batch_peer_bytes(dmf_batch_t b, int32_t world, size_t* bytes) {
    if (!b || !bytes || world < 1) return fail(DMF_E_ARG, "bad argument");
    if (!b->p.gram_ok) return fail(DMF_E_SHAPE, "no Gram-engine instantiation for this shape");
    const size_t slot = b->p.per_fit_stats / 8 * b->shape.n_fits;
    *bytes = align_up(2 * (size_t)world * slot * 8, 256) + align_up(2 * (size_t)world * 4, 256);
    return DMF_OK;
}
int dmf_batch_set_peers(dmf_batch_t b, int32_t rank, int32_t world, const void* const* peer_bases, size_t bytes_per_peer, void* stream) {
    if (!b || !peer_bases || world < 1 || rank < 0 || rank >= world || world > kThreads) return fail(DMF_E_ARG, "bad argument");
    if (!b->sharded) return fail(DMF_E_STATE, "peer exchange belongs to row-sharded batches (dmf_batch_set_sharded first)");
    size_t need = 0;
    int rc = dmf_batch_peer_bytes(b, world, &need);
    if (rc) return rc;
    if (bytes_per_peer < need) return fail(DMF_E_ARG, "symmetric buffers too small (dmf_batch_peer_bytes)");
    for (int r = 0; r < world; ++r)
        if (!peer_bases[r] || (reinterpret_cast<uintptr_t>(peer_bases[r]) & 15)) return fail(DMF_E_ARG, "peer buffer pointers must be non-NULL and 16-byte aligned");
    cudaStream_t st = (cudaStream_t)stream;
    if (!b->peers_dev) CUDA_TRY(cudaMalloc(&b->peers_dev, sizeof(double*) * kThreads));
    if (!b->xchg_ticket) CUDA_TRY(cudaMalloc(&b->xchg_ticket, 256));
    CUDA_TRY(cudaMemcpyAsync(b->peers_dev, peer_bases, sizeof(double*) * world, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(b->xchg_ticket, 0, 256, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    b->peer_rank = rank; b->peer_world = world;
    b->peer_slot_stride = (long long)(b->p.per_fit_stats / 8 * b->shape.n_fits);
    b->peer_flag_off = (long long)align_up(2 * (size_t)world * b->peer_slot_stride * 8, 256);
    b->xchg_epoch = 0;      // the caller zeroes the symmetric buffers (flags) before the first exchange
    return DMF_OK;
}
int dmf_gram_exchange(dmf_batch_t b, int32_t which, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->peers_dev || b->peer_world < 1) return fail(DMF_E_STATE, "dmf_batch_set_peers first");
    if (which < 0 || which > 2) return fail(DMF_E_ARG, "which must be 0 (blocks), 1 (scalars) or 2 (scalars at set-up)");
    XchgArgs a;
    a.peers = b->peers_dev;
    a.local = b->stats_local; a.global = b->stats_global;
    a.ticket = b->xchg_ticket;
    a.per_fit = (long long)(b->p.per_fit_stats / 8); a.slot_stride = b->peer_slot_stride; a.flag_off = b->peer_flag_off;
    a.scal_off = (long long)b->p.stats_scal;
    a.n_fits = b->shape.n_fits; a.rank = b->peer_rank; a.world = b->peer_world; a.which = which;
    a.epoch_dev = b->xchg_ticket + 16;            // the exchange count lives on the device: CUDA-graph replays advance it
    ++b->xchg_epoch;
    const long long n = which == 0 ? (long long)a.n_fits * a.per_fit : (long long)a.n_fits * 8;
    const int ctas = (int)std::max<long long>(1, std::min<long long>(32, (n + kThreads * 4 - 1) / (kThreads * 4)));
    peer_allreduce_kernel<<<ctas, kThreads, 0, (cudaStream_t)stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    b->launches++;
    return DMF_OK;
}

int dmf_batch_reserve_momentum(dmf_batch_t b, int64_t n_inner_total, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (n_inner_total < 0) return fail(DMF_E_ARG, "negative iteration count");
    return ensure_mom(b, n_inner_total, (cudaStream_t)stream);
}

int dmf_gram_init(dmf_batch_t b, void* stream) {
    int rc = dmf_gram_rowgram(b, 1, 0.0, stream);
    if (rc) return rc;
    return b->shape.K ? dmf_gram_panels(b, 1, stream) : DMF_OK;
}
int dmf_gram_outer(dmf_batch_t b, int32_t n_iter2, double tol, void* stream) {
    int rc;
    if (n_iter2 > 0) {
        if ((rc = dmf_gram_u_inner(b, n_iter2, stream))) return rc;
        if ((rc = dmf_gram_panels(b, 0, stream))) return rc;
        if ((rc = dmf_gram_alpha_inner(b, n_iter2, stream))) return rc;
    }
    return dmf_gram_rowgram(b, 0, tol, stream);
}

int dmf_fused_pass(dmf_batch_t b, int32_t n_iter2, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->p.fused_ok) return fail(DMF_E_SHAPE, "no fused-engine instantiation for this shape / layout");
    if (b->multmode) return fail(DMF_E_STATE, "the fused engine does not run multiplicity-form batches");
    if (n_iter2 < 1 || n_iter2 > kFusedMaxInner) return fail(DMF_E_ARG, "the fused pass runs 1 .. 64 update_u iterations per visit");
    b->t_hi += n_iter2;
    int rc = ensure_mom(b, b->t_hi + n_iter2, (cudaStream_t)stream);
    if (rc) return rc;
    const Plan& p = b->p;
    fused_kern_t k = by_types_f(b->shape, p.kb_f, p.nub_f, p.s_f);
    FusedArgs a = p.fa;
    a.fits = b->fits_dev;
    a.n_iter2 = n_iter2;
    a.flags = b->sharded ? kFlagPartial : 0;      // row-sharded: publish this GPU's sums, dmf_fused_alpha_commit decides on the reduced ones
    a.tol = tol;
    a.mom_a = b->mom_dev; a.mom_m = b->mom_dev + b->mom_cap;
    k<<<dim3(a.g.n_parts, b->n_active, 1), p.fc.threads, p.smem_f, (cudaStream_t)stream>>>(a);
    CUDA_TRY(cudaGetLastError());
    b->launches++;
    b->fused_pending = 1;
    return DMF_OK;
}
int dmf_fused_outer(dmf_batch_t b, int32_t n_iter2, double tol, void* stream) {
    if (b && b->sharded) return fail(DMF_E_STATE, "row-sharded batches: dmf_fused_pass, all-reduce of the statistics blocks, dmf_fused_alpha_commit");
    int rc = dmf_fused_pass(b, n_iter2, tol, stream);
    if (rc) return rc;
    return dmf_gram_alpha_inner(b, n_iter2, stream);
}
int dmf_fused_alpha_commit(dmf_batch_t b, int32_t n_iter2, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->sharded || !b->p.fused_ok) return fail(DMF_E_STATE, "dmf_fused_alpha_commit follows dmf_fused_pass on a row-sharded batch");
    if (n_iter2 < 0) return fail(DMF_E_ARG, "negative iteration count");
    int rc = ensure_mom(b, b->t_hi + n_iter2, (cudaStream_t)stream);
    if (rc) return rc;
    return launch_g(b, k_ainner(b), b->p.ntc_p, 0, (b->shape.mode == DMF_MODE_PURITY ? kFlagFW : 0) | kFlagFusedCommit, n_iter2, tol, 0, 0, 0, 1,
                    (cudaStream_t)stream);
}
int dmf_fused_finish(dmf_batch_t b, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (!b->fused_pending) return DMF_OK;
    b->fused_pending = 0;
    return dmf_gram_rowgram(b, 0, tol, stream);          // cost-only use of the rowgram pass: counts the outer iteration, runs the test
}

// engine actually used for a call with n_iter2 inner iterations
static int effective_engine(const dmf_batch_s* b, int n_iter2) {
    if (b->engine == DMF_ENGINE_FUSED && (n_iter2 < 1 || n_iter2 > kFusedMaxInner || b->sharded || b->multmode)) return DMF_ENGINE_GRAM;      // (sharded fits are driven step by step by the caller)
    return b->engine;
}

int dmf_enqueue_outer(dmf_batch_t b, int32_t n_outer, int32_t n_iter2, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    int rc;
    const int eng = effective_engine(b, n_iter2);
    if (eng == DMF_ENGINE_FUSED) {        // leaves the cost of the last iterate pending: dmf_fused_finish
        for (int o = 0; o < n_outer; ++o)
            if ((rc = dmf_fused_outer(b, n_iter2, tol, stream))) return rc;
        return DMF_OK;
    }
    if (b->fused_pending && (rc = dmf_fused_finish(b, tol, stream))) return rc;
    if (eng == DMF_ENGINE_GRAM) {
        for (int o = 0; o < n_outer; ++o)
            if ((rc = dmf_gram_outer(b, n_iter2, tol, stream))) return rc;
        return DMF_OK;
    }
    for (int o = 0; o < n_outer; ++o) {
        for (int i = 0; i < n_iter2; ++i)
            if ((rc = dmf_pass_u(b, stream))) return rc;
        for (int i = 0; i < n_iter2; ++i)
            if ((rc = (b->shape.mode == DMF_MODE_PURITY) ? dmf_pass_fw(b, i, stream) : dmf_pass_alpha(b, stream))) return rc;
        if ((rc = dmf_pass_cost(b, tol, stream))) return rc;
    }
    return DMF_OK;
}

int dmf_batch_read_state(dmf_batch_t b, dmf_fit_state_t* out, int32_t n, void* stream) {
    if (!b || !out) return fail(DMF_E_ARG, "NULL argument");
    if (n > b->shape.n_fits) n = b->shape.n_fits;
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemcpyAsync(b->pinned, b->states_dev, sizeof(FitState) * n, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int i = 0; i < n; ++i) {
        const FitState& s = b->pinned[i];
        out[i].cost = s.cf; out[i].cost_prev = s.cf_prev; out[i].l_w = s.l_w; out[i].l_h = s.l_h;
        out[i].a1 = s.a1; out[i].a2 = s.a2; out[i].dmax = s.dmax;
        out[i].n_outer = s.n_outer; out[i].done = s.done; out[i].u_slot = s.u_cur; out[i].a_slot = s.a_cur;
    }
    return DMF_OK;
}

int dmf_fit_batched(dmf_batch_t b, int32_t n_iter1, int32_t n_iter2, double tol, void* stream) {
    if (!b) return fail(DMF_E_ARG, "NULL batch");
    if (n_iter1 < 0 || n_iter2 < 0) return fail(DMF_E_ARG, "negative iteration count");
    cudaStream_t st = (cudaStream_t)stream;
    const int eng = effective_engine(b, n_iter2);
    b->fused_pending = 0;
    int rc = eng != DMF_ENGINE_STREAM ? dmf_gram_init(b, stream) : dmf_pass_init(b, stream);
    if (rc) return rc;
    // Outer iterations are enqueued in chunks; after each chunk the per-fit `done` flags come back through
    // pinned memory.  Terminated fits skip their launches on the device, so over-enqueueing is harmless.
    int issued = 0, chunk = 2;
    const int n = b->shape.n_fits;
    while (issued < n_iter1) {
        const int todo = std::min(chunk, n_iter1 - issued);
        if ((rc = dmf_enqueue_outer(b, todo, n_iter2, tol, stream))) return rc;
        issued += todo;
        if (issued == n_iter1 && eng == DMF_ENGINE_FUSED && (rc = dmf_fused_finish(b, tol, stream))) return rc;    // cost of the last iterate
        CUDA_TRY(cudaMemcpyAsync(b->pinned, b->states_dev, sizeof(FitState) * n, cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaStreamSynchronize(st));
        std::vector<int> active;
        for (int i = 0; i < n; ++i) {
            if (b->pinned[i].done == 3) return fail(DMF_E_STATE, "non-finite values reached the simplex projection (fit " + std::to_string(i) + ")");
            if (b->pinned[i].done == 0) active.push_back(i);
        }
        if (active.empty()) { b->fused_pending = 0; break; }
        // launch only the still-running fits from now on (terminated fits would return at once, but their CTAs still cost a launch slot)
        if ((int)active.size() != b->n_active && (rc = upload_fits(b, &active, st))) return rc;
        chunk = std::min(chunk * 2, 16);
    }
    CUDA_TRY(cudaStreamSynchronize(st));
    return DMF_OK;
}

int dmf_batch_launch_count(dmf_batch_t b, int64_t* out) {
    if (!b || !out) return fail(DMF_E_ARG, "NULL argument");
    *out = b->launches;
    return DMF_OK;
}

int dmf_pack_weights_u16(const void* src, int32_t kind, int64_t count, uint16_t* dst, int32_t* bad_dev, void* stream) {
    if (!src || !dst || !bad_dev || count < 0) return fail(DMF_E_ARG, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(bad_dev, 0, sizeof(int32_t), st));
    if (count == 0) return DMF_OK;
    const int threads = 256;
    const int blocks = (int)std::min<long long>((count + threads - 1) / threads, 148 * 16);
    if (kind == 0) pack_u16_kernel<double><<<blocks, threads, 0, st>>>((const double*)src, count, dst, bad_dev);
    else if (kind == 1) pack_u16_kernel<float><<<blocks, threads, 0, st>>>((const float*)src, count, dst, bad_dev);
    else if (kind == 2) pack_u16_kernel<long long><<<blocks, threads, 0, st>>>((const long long*)src, count, dst, bad_dev);
    else return fail(DMF_E_ARG, "src_kind must be 0 (f64), 1 (f32) or 2 (i64)");
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

int dmf_gather_rows(const void* src, const int32_t* rows, int64_t n_rows, int64_t row_elems, int32_t elem_bytes, void* dst, void* stream) {
    if (!src || !rows || !dst || n_rows < 0 || row_elems <= 0) return fail(DMF_E_ARG, "bad argument");
    if (elem_bytes != 1 && elem_bytes != 2 && elem_bytes != 4 && elem_bytes != 8) return fail(DMF_E_ARG, "elem_bytes must be 1, 2, 4 or 8");
    if (n_rows == 0) return DMF_OK;
    const int threads = 256;
    const int blocks = (int)std::min<long long>((n_rows * 32 + threads - 1) / threads, 148 * 16);
    gather_rows_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>((const char*)src, rows, n_rows, row_elems * elem_bytes, (char*)dst);
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

}  // extern "C"

// =================================================================================================
// wls_intercept for all samples (dmf_wls.cuh)
#include "dmf_wls.cuh"

namespace {

struct WlsPlan {
    int slab, ntc, rg, tile_rows, n_tiles, n_parts, n_groups, part_stride, Kz, nblk;
    StageLayout stage;    // X, D, R1, R2
    unsigned smem;
    size_t off_fit, off_tickets, off_part, off_gpart, off_mom, off_status, ws_bytes;
};

int make_wls_plan(const dmf_handle_s* h, const dmf_wls_desc_t& d, WlsPlan& p) {
    if (d.M <= 0 || d.N <= 0 || d.K < 0 || d.K2 < 0 || d.K + d.K2 <= 0) return fail(DMF_E_SHAPE, "wls: M, N positive and K + K2 >= 1 required");
    if (d.K + d.K2 > kMaxKt) return fail(DMF_E_SHAPE, "wls: more than 32 regressors are not supported by this build");
    if (d.dtype != DMF_F64 && d.dtype != DMF_F32) return fail(DMF_E_ARG, "dtype must be DMF_F64 or DMF_F32");
    if (d.wtype != DMF_W_FLOAT && d.wtype != DMF_W_U16) return fail(DMF_E_ARG, "wtype must be DMF_W_FLOAT or DMF_W_U16");
    if (d.ldx < d.N || d.ldd < d.N || (d.K && d.ldr < d.K) || (d.K2 && d.ldr2 < d.K2)) return fail(DMF_E_SHAPE, "wls: row pitch smaller than the row");
    if ((d.ldx | d.ldd | (d.K ? d.ldr : 0) | (d.K2 ? d.ldr2 : 0)) & 1) return fail(DMF_E_SHAPE, "wls: row pitches must be even (zero padded)");
    const size_t sT = d.dtype == DMF_F64 ? 8 : 4, sW = d.wtype == DMF_W_U16 ? 2 : sT;
    p.slab = std::min<int>(d.N, kConsumers);            // sample columns per launch (one column per thread)
    p.ntc = pow2ceil(p.slab);
    p.rg = kConsumers / p.ntc;
    const size_t px = d.ldx * sT, pd = d.ldd * sW, pr = d.K ? d.ldr * sT : 0, pu = d.K2 ? d.ldr2 * sT : 0;
    int ra = 1;
    while (ra < 16 && ((ra * px) % 16 || (ra * pd) % 16 || (ra * pr) % 16 || (ra * pu) % 16)) ra <<= 1;
    const size_t budget = std::min<size_t>((size_t)h->max_smem_optin, 200 * 1024) - kCtlBytes - 2048;
    const size_t rows_w[kMaxSrc] = {px, pd, pr, pu, 0};
    long long tr = 0;
    for (long long cand = (long long)p.rg * 8; cand >= 1; cand >>= 1) {
        if (cand % ra) continue;
        if (stage_layout(cand, rows_w, rows_w).bytes * kStages <= budget) { tr = cand; break; }
    }
    if (!tr) return fail(DMF_E_SHAPE, "wls: one row tile does not fit in shared memory");
    p.tile_rows = (int)tr;
    p.n_tiles = (int)((d.M + tr - 1) / tr);
    p.stage = stage_layout(tr, rows_w, rows_w);
    p.n_parts = std::min(p.n_tiles, h->sm_count);
    p.n_groups = (p.n_parts + kGroup - 1) / kGroup;
    p.part_stride = kWlsBlock * kWlsBlock * p.slab;
    p.Kz = d.K + d.K2 + 2;
    p.nblk = (p.Kz + kWlsBlock - 1) / kWlsBlock;
    p.smem = (unsigned)std::max<size_t>(kCtlBytes + (size_t)kStages * p.stage.bytes, kCtlBytes + (size_t)p.part_stride * 8 + 256);
    if (p.smem > (unsigned)h->max_smem_optin) return fail(DMF_E_SHAPE, "wls: shared-memory plan exceeds the device limit");
    p.off_fit = 0;
    p.off_tickets = 256;
    p.off_part = align_up(p.off_tickets + sizeof(unsigned) * (p.n_groups + 1), 256);
    p.off_gpart = align_up(p.off_part + (size_t)p.n_parts * p.part_stride * 8, 256);
    p.off_mom = align_up(p.off_gpart + (size_t)p.n_groups * p.part_stride * 8, 256);
    p.off_status = align_up(p.off_mom + (size_t)p.Kz * p.Kz * p.slab * 8, 256);
    p.ws_bytes = p.off_status + 256;
    return DMF_OK;
}

wls_kern_t wls_kernel_of(const dmf_wls_desc_t& d) {
    return d.dtype == DMF_F64 ? (d.wtype == DMF_W_U16 ? pick_wls_f64_u16() : pick_wls_f64_f64())
                              : (d.wtype == DMF_W_U16 ? pick_wls_f32_u16() : pick_wls_f32_f32());
}

// workspace checks and kernel attribute of one dmf_wls_fit / dmf_wls_moments call
int wls_prepare(const dmf_handle_s* h, const dmf_wls_desc_t* dd, void* ws, size_t ws_bytes, void* stream, WlsPlan& p) {
    if (!h || !dd || !ws) return fail(DMF_E_ARG, "NULL argument");
    const dmf_wls_desc_t& d = *dd;
    if (!d.X || !d.D || !d.out || (d.K && !d.R1) || (d.K2 && !d.R2)) return fail(DMF_E_ARG, "wls: NULL matrix");
    int rc = make_wls_plan(h, d, p);
    if (rc) return rc;
    if (ws_bytes < p.ws_bytes) return fail(DMF_E_ARG, "wls: workspace too small");
    if (reinterpret_cast<uintptr_t>(ws) & 255) return fail(DMF_E_ARG, "workspace must be 256-byte aligned");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    char* base = static_cast<char*>(ws);
    CUDA_TRY(cudaFuncSetAttribute((const void*)wls_kernel_of(d), cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    CUDA_TRY(cudaMemsetAsync(base + p.off_tickets, 0, p.off_part - p.off_tickets, st));
    CUDA_TRY(cudaMemsetAsync(base + p.off_status, 0, 256, st));
    return DMF_OK;
}

// the moment launches of sample columns j0 .. j0 + ns into the workspace's [Kz Kz][ns] matrix
int wls_moments_slab(const dmf_wls_desc_t& d, const WlsPlan& p, char* base, int j0, int ns, cudaStream_t st) {
    const size_t sT = d.dtype == DMF_F64 ? 8 : 4, sW = d.wtype == DMF_W_U16 ? 2 : sT;
    FitDev f;
    memset(&f, 0, sizeof(f));
    f.X = static_cast<const char*>(d.X) + (size_t)j0 * sT;
    f.D = static_cast<const char*>(d.D) + (size_t)j0 * sW;
    f.Rk = static_cast<const char*>(d.R1);
    f.U = const_cast<char*>(static_cast<const char*>(d.R2));
    f.part = reinterpret_cast<double*>(base + p.off_part);
    f.gpart = reinterpret_cast<double*>(base + p.off_gpart);
    f.tickets = reinterpret_cast<unsigned*>(base + p.off_tickets);
    CUDA_TRY(cudaMemcpyAsync(base + p.off_fit, &f, sizeof(f), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));   // `f` is a stack temporary
    WlsArgs a;
    memset(&a, 0, sizeof(a));
    Geom& g = a.g;
    g.M = d.M; g.N = ns; g.K = d.K; g.nu = d.K2; g.Kt = d.K + d.K2;
    g.ldx = d.ldx; g.ldd = d.ldd; g.ldr = d.K ? d.ldr : 0; g.ldu = d.K2 ? d.ldr2 : 0;
    g.tile_rows = p.tile_rows; g.n_tiles = p.n_tiles; g.ntc = pow2ceil(ns); g.rg = kConsumers / g.ntc;
    // rows of a tile are walked with stride rg: a narrower last slab only changes the thread mapping
    g.n_parts = p.n_parts; g.n_groups = p.n_groups; g.part_stride = p.part_stride;
    set_stages(g, p.stage);
    g.offUp = g.offU;
    a.fits = reinterpret_cast<const FitDev*>(base + p.off_fit);
    a.mom = reinterpret_cast<double*>(base + p.off_mom);
    a.Kfull = d.K + d.K2;
    a.y_is_dx = d.y_is_dx;
    const wls_kern_t kern = wls_kernel_of(d);
    for (int bi = 0; bi < p.nblk; ++bi)
        for (int bj = bi; bj < p.nblk; ++bj) {
            a.bi = bi; a.bj = bj;
            kern<<<dim3(p.n_parts, 1, 1), kThreads, p.smem, st>>>(a);
            CUDA_TRY(cudaGetLastError());
        }
    return DMF_OK;
}

// reads the NNLS status word (synchronises the stream)
int wls_status(const void* status_dev, cudaStream_t st) {
    int status = 0;
    CUDA_TRY(cudaMemcpyAsync(&status, status_dev, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    if (status & 1) return fail(DMF_E_STATE, "wls: a sample produced non-finite proportions (all of its weights zero, or non-finite inputs)");
    if (status & 2) return fail(DMF_E_STATE, "wls: the regressors of a sample are collinear (non-positive pivot in the normal equations)");
    return DMF_OK;
}

}  // namespace

extern "C" {

int dmf_wls_workspace_bytes(dmf_handle_t h, const dmf_wls_desc_t* d, size_t* bytes) {
    if (!h || !d || !bytes) return fail(DMF_E_ARG, "NULL argument");
    WlsPlan p;
    int rc = make_wls_plan(h, *d, p);
    if (rc) return rc;
    *bytes = p.ws_bytes;
    return DMF_OK;
}

int dmf_wls_fit(dmf_handle_t h, const dmf_wls_desc_t* dd, void* ws, size_t ws_bytes, void* stream) {
    WlsPlan p;
    int rc = wls_prepare(h, dd, ws, ws_bytes, stream, p);
    if (rc) return rc;
    const dmf_wls_desc_t& d = *dd;
    cudaStream_t st = (cudaStream_t)stream;
    char* base = static_cast<char*>(ws);
    for (int j0 = 0; j0 < d.N; j0 += p.slab) {
        const int ns = std::min(p.slab, d.N - j0);
        rc = wls_moments_slab(d, p, base, j0, ns, st);
        if (rc) return rc;
        wls_nnls_kernel<<<(ns + 63) / 64, 64, 0, st>>>(reinterpret_cast<double*>(base + p.off_mom), d.K + d.K2, ns, d.M, d.out + j0,
                                                      (long long)d.N, reinterpret_cast<int*>(base + p.off_status));
        CUDA_TRY(cudaGetLastError());
    }
    return wls_status(base + p.off_status, st);
}

int dmf_wls_moments(dmf_handle_t h, const dmf_wls_desc_t* dd, double* mom, void* ws, size_t ws_bytes, void* stream) {
    if (!h || !dd || !mom) return fail(DMF_E_ARG, "NULL argument");
    const dmf_wls_desc_t& d = *dd;
    cudaStream_t st = (cudaStream_t)stream;
    const size_t Kz = (size_t)(d.K + d.K2 + 2);
    if (d.M == 0 && d.N > 0 && d.K >= 0 && d.K2 >= 0) {      // a GPU that holds no rows contributes zero moments
        CUDA_TRY(cudaSetDevice(h->device));
        CUDA_TRY(cudaMemsetAsync(mom, 0, Kz * Kz * d.N * sizeof(double), st));
        return DMF_OK;
    }
    WlsPlan p;
    int rc = wls_prepare(h, dd, ws, ws_bytes, stream, p);
    if (rc) return rc;
    char* base = static_cast<char*>(ws);
    for (int j0 = 0; j0 < d.N; j0 += p.slab) {
        const int ns = std::min(p.slab, d.N - j0);
        rc = wls_moments_slab(d, p, base, j0, ns, st);
        if (rc) return rc;
        // the slab's [Kz Kz][ns] block into columns j0 .. j0 + ns of the caller's [Kz Kz][N] matrix
        CUDA_TRY(cudaMemcpy2DAsync(mom + j0, d.N * sizeof(double), base + p.off_mom, ns * sizeof(double), ns * sizeof(double), Kz * Kz,
                                   cudaMemcpyDeviceToDevice, st));
    }
    return DMF_OK;
}

int dmf_wls_solve(dmf_handle_t h, const dmf_wls_desc_t* dd, const double* mom, void* ws, size_t ws_bytes, void* stream) {
    if (!h || !dd || !mom || !ws) return fail(DMF_E_ARG, "NULL argument");
    const dmf_wls_desc_t& d = *dd;
    if (!d.out) return fail(DMF_E_ARG, "wls: NULL matrix");
    if (d.M <= 0 || d.N <= 0 || d.K < 0 || d.K2 < 0 || d.K + d.K2 <= 0) return fail(DMF_E_SHAPE, "wls: M, N positive and K + K2 >= 1 required");
    if (d.K + d.K2 > kMaxKt) return fail(DMF_E_SHAPE, "wls: more than 32 regressors are not supported by this build");
    if (ws_bytes < 256) return fail(DMF_E_ARG, "wls: workspace too small");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaMemsetAsync(ws, 0, 256, st));
    // one thread per sample reads column j of the [Kz Kz][N] matrix: the same moments, K and M as dmf_wls_fit's per-slab launches
    wls_nnls_kernel<<<(d.N + 63) / 64, 64, 0, st>>>(mom, d.K + d.K2, d.N, d.M, d.out, (long long)d.N, static_cast<int*>(ws));
    CUDA_TRY(cudaGetLastError());
    return wls_status(ws, st);
}

}  // extern "C"

// =================================================================================================
// the steps right before / after the path (dmf_post.cuh)
#include "dmf_post.cuh"

extern "C" {

int dmf_nndsvd_split(const double* U, int64_t ldu, const double* S, const double* Vh, int64_t ldv, int64_t M, int32_t N, int32_t rank,
                     double* W, double* H, void* stream) {
    if (!U || !S || !Vh || !W || !H || M <= 0 || N <= 0 || rank <= 0 || ldu < rank || ldv < N) return fail(DMF_E_ARG, "nndsvd: bad argument");
    nndsvd_split_kernel<<<rank, 256, 0, (cudaStream_t)stream>>>(U, ldu, S, Vh, ldv, M, N, rank, W, H);
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

int dmf_percentile_max_keep(void) { return 128; }

int dmf_percentile_bounds(const double* stack, int32_t B, int64_t P, double q_lo, double q_hi, double* out_lo, double* out_hi, void* stream) {
    if (!stack || !out_lo || !out_hi || B <= 0 || P < 0) return fail(DMF_E_ARG, "percentile: bad argument");
    if (!(q_lo >= 0.0 && q_lo <= q_hi && q_hi <= 100.0)) return fail(DMF_E_ARG, "percentile: 0 <= q_lo <= q_hi <= 100 required");
    if (P == 0) return DMF_OK;
    const int klo = (int)floor((double)(B - 1) * (q_lo / 100.0)), khi = (int)floor((double)(B - 1) * (q_hi / 100.0));
    const int keep = std::max(std::min(klo + 2, B), std::min(B - khi, B));
    const int blocks = (int)((P + 127) / 128);
    if (keep <= 32) percentile_kernel<32><<<blocks, 128, 0, (cudaStream_t)stream>>>(stack, B, P, q_lo, q_hi, out_lo, out_hi);
    else if (keep <= 128) percentile_kernel<128><<<blocks, 128, 0, (cudaStream_t)stream>>>(stack, B, P, q_lo, q_hi, out_lo, out_hi);
    else return fail(DMF_E_SHAPE, "percentile: more than 128 order statistics per tail would have to be kept (dmf_percentile_max_keep)");
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

int dmf_rng_legacy_streams(const uint32_t* seeds, int32_t n_streams, int64_t M, int32_t* idx, int64_t ld_idx, int64_t n_dbl, double* u,
                           int64_t ld_u, uint32_t* state, void* stream) {
    if (!seeds || n_streams < 0 || M < 0 || n_dbl < 0) return fail(DMF_E_ARG, "rng: bad argument");
    if (M > 0x7fffffffll) return fail(DMF_E_ARG, "rng: row indices are int32 (M < 2^31)");
    if ((idx && ld_idx < M) || (u && ld_u < n_dbl)) return fail(DMF_E_ARG, "rng: output pitch smaller than the row");
    if (n_streams == 0 || (!idx && !u && !state)) return DMF_OK;
    legacy_streams_kernel<<<dim3((n_streams + kRngWarps - 1) / kRngWarps, 2, 1), kRngWarps * 32, 0, (cudaStream_t)stream>>>(
        seeds, n_streams, (long long)M, idx, (long long)ld_idx, (long long)n_dbl, u, (long long)ld_u, state);
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

int dmf_consensus(const double* alpha_runs, int32_t n_runs, int32_t Kt, int32_t N, int32_t* labels_ws, double* consensus, void* stream) {
    if (!alpha_runs || !labels_ws || !consensus || n_runs <= 0 || Kt <= 0 || N <= 0) return fail(DMF_E_ARG, "consensus: bad argument");
    labels_kernel<<<(n_runs * N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(alpha_runs, n_runs, Kt, N, labels_ws);
    CUDA_TRY(cudaGetLastError());
    const long long nn = (long long)N * N;
    consensus_kernel<<<(int)((nn + 127) / 128), 128, 0, (cudaStream_t)stream>>>(labels_ws, n_runs, N, consensus);
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

}  // extern "C"

// =================================================================================================
// NNDSVD of the floored residual over row-sharded rows (dmf_resid.cuh)
#include "dmf_resid.cuh"

namespace {

struct ResidPlan {
    int nt, n_tri, tile_rows, n_tiles, n_parts, n_groups, stages;   // resid_gram_kernel
    int p_parts, p_groups;                                          // resid_project_kernel
    StageLayout stage;
    unsigned smem;
    size_t off_fits, off_tickets, off_part, off_gpart, off_pfit, off_ptickets, off_ppart, off_pgpart, ws_bytes;
};

int make_resid_plan(const dmf_handle_s* h, const dmf_resid_desc_t& d, ResidPlan& p) {
    if (d.M < 0 || d.N <= 0 || d.K < 0) return fail(DMF_E_SHAPE, "resid: M >= 0, N > 0 and K >= 0 required");
    if (d.N > kMaxResidN) return fail(DMF_E_SHAPE, "resid: more than 512 samples are not supported by this build");
    if (d.K > kMaxKt) return fail(DMF_E_SHAPE, "resid: more than 32 reference columns are not supported by this build");
    if (d.ldx < d.N || (d.K && d.ldr < d.K) || ((d.ldx | (d.K ? d.ldr : 0)) & 1))
        return fail(DMF_E_SHAPE, "resid: row pitches must be even and at least the row");
    p.nt = (d.N + kGramTile - 1) / kGramTile;
    p.n_tri = p.nt * (p.nt + 1) / 2;
    const size_t rows_w[kMaxSrc] = {(size_t)d.ldx * 8, 0, d.K ? (size_t)d.ldr * 8 : 0, 0, 0};
    const size_t budget = (size_t)h->max_smem_optin - kCtlBytes;
    p.tile_rows = 0;
    for (int tr = kResMaxRows; tr >= 4 && !p.tile_rows; tr >>= 1)
        for (int stg = kStages; stg >= 3; --stg) {
            const size_t ring = std::max<size_t>(stage_layout(tr, rows_w, rows_w).bytes * stg, (size_t)kGramTile * kGramTile * 8);
            if (ring + (size_t)tr * kResPitch * 8 <= budget) { p.tile_rows = tr; p.stages = stg; break; }
        }
    if (!p.tile_rows) return fail(DMF_E_SHAPE, "resid: one row tile does not fit in shared memory");
    p.stage = stage_layout(p.tile_rows, rows_w, rows_w);
    p.smem = (unsigned)(kCtlBytes + std::max<size_t>((size_t)p.stage.bytes * p.stages, (size_t)kGramTile * kGramTile * 8) +
                        (size_t)p.tile_rows * kResPitch * 8);
    p.n_tiles = (int)std::max<long long>(1, (d.M + p.tile_rows - 1) / p.tile_rows);
    // two CTAs per SM over all G tiles, never more row splits than row tiles
    p.n_parts = std::max(1, std::min(p.n_tiles, 2 * h->sm_count / p.n_tri));
    p.n_groups = groups_of(p.n_parts);
    p.p_parts = (int)std::max<long long>(1, std::min<long long>((d.M + 7) / 8, 4LL * h->sm_count));
    p.p_groups = groups_of(p.p_parts);
    const size_t TT = (size_t)kGramTile * kGramTile;
    p.off_fits = 0;
    p.off_tickets = align_up(sizeof(FitDev) * p.n_tri, 256);
    p.off_part = align_up(p.off_tickets + sizeof(unsigned) * p.n_tri * (p.n_groups + 1), 256);
    p.off_gpart = align_up(p.off_part + (size_t)p.n_tri * p.n_parts * TT * 8, 256);
    p.off_pfit = align_up(p.off_gpart + (size_t)p.n_tri * p.n_groups * TT * 8, 256);
    p.off_ptickets = align_up(p.off_pfit + sizeof(FitDev), 256);
    p.off_ppart = align_up(p.off_ptickets + sizeof(unsigned) * (p.p_groups + 1), 256);
    p.off_pgpart = align_up(p.off_ppart + (size_t)p.p_parts * 2 * kMaxKt * 8, 256);
    p.ws_bytes = align_up(p.off_pgpart + (size_t)p.p_groups * 2 * kMaxKt * 8, 256);
    return DMF_OK;
}

int resid_check(const dmf_handle_s* h, const dmf_resid_desc_t* d, void* ws, size_t ws_bytes, ResidPlan& p) {
    if (!h || !d || !ws) return fail(DMF_E_ARG, "NULL argument");
    if ((d->M && !d->X) || (d->M && d->K && (!d->R || !d->H1))) return fail(DMF_E_ARG, "resid: NULL matrix");
    int rc = make_resid_plan(h, *d, p);
    if (rc) return rc;
    if (ws_bytes < p.ws_bytes) return fail(DMF_E_ARG, "resid: workspace too small");
    if (reinterpret_cast<uintptr_t>(ws) & 255) return fail(DMF_E_ARG, "workspace must be 256-byte aligned");
    return DMF_OK;
}

}  // namespace

extern "C" {

int dmf_resid_workspace_bytes(dmf_handle_t h, const dmf_resid_desc_t* d, size_t* bytes) {
    if (!h || !d || !bytes) return fail(DMF_E_ARG, "NULL argument");
    ResidPlan p;
    int rc = make_resid_plan(h, *d, p);
    if (rc) return rc;
    *bytes = p.ws_bytes;
    return DMF_OK;
}

int dmf_resid_gram(dmf_handle_t h, const dmf_resid_desc_t* d, double* G, int32_t* has_negative, void* ws, size_t ws_bytes, void* stream) {
    ResidPlan p;
    int rc = resid_check(h, d, ws, ws_bytes, p);
    if (rc) return rc;
    if (!G || !has_negative) return fail(DMF_E_ARG, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    char* base = static_cast<char*>(ws);
    CUDA_TRY(cudaMemsetAsync(has_negative, 0, sizeof(int32_t), st));
    if (d->M == 0) {                                     // a GPU that holds no rows contributes zero
        CUDA_TRY(cudaMemsetAsync(G, 0, (size_t)d->N * d->N * sizeof(double), st));
        return DMF_OK;
    }
    const size_t TT = (size_t)kGramTile * kGramTile;
    std::vector<FitDev> fits(p.n_tri);
    for (int t = 0; t < p.n_tri; ++t) {
        FitDev& f = fits[t];
        memset(&f, 0, sizeof(f));
        f.X = reinterpret_cast<const char*>(d->X);
        f.Rk = d->K ? reinterpret_cast<const char*>(d->R) : nullptr;
        f.part = reinterpret_cast<double*>(base + p.off_part) + (size_t)t * p.n_parts * TT;
        f.gpart = reinterpret_cast<double*>(base + p.off_gpart) + (size_t)t * p.n_groups * TT;
        f.tickets = reinterpret_cast<unsigned*>(base + p.off_tickets) + (size_t)t * (p.n_groups + 1);
    }
    CUDA_TRY(cudaMemcpyAsync(base + p.off_fits, fits.data(), sizeof(FitDev) * p.n_tri, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(base + p.off_tickets, 0, p.off_part - p.off_tickets, st));
    ResidArgs a;
    memset(&a, 0, sizeof(a));
    Geom& g = a.g;
    g.M = d->M; g.N = d->N; g.K = d->K;
    g.ldx = d->ldx; g.ldr = d->K ? d->ldr : 0;
    g.tile_rows = p.tile_rows; g.n_tiles = p.n_tiles;
    g.n_parts = p.n_parts; g.n_groups = p.n_groups; g.part_stride = (int)TT;
    g.stages = p.stages;
    set_stages(g, p.stage);
    a.fits = reinterpret_cast<const FitDev*>(base + p.off_fits);
    a.H1 = d->H1;
    a.G = G;
    a.neg = has_negative;
    a.nt = p.nt;
    CUDA_TRY(cudaFuncSetAttribute((const void*)resid_gram_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
    resid_gram_kernel<<<dim3(p.n_parts, p.n_tri, 1), kThreads, p.smem, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));                 // `fits` is a host temporary
    return DMF_OK;
}

int dmf_resid_project(dmf_handle_t h, const dmf_resid_desc_t* d, const double* Vh, const double* inv_sigma, int32_t rank, double* U,
                      double* sums, void* ws, size_t ws_bytes, void* stream) {
    ResidPlan p;
    int rc = resid_check(h, d, ws, ws_bytes, p);
    if (rc) return rc;
    if (rank <= 0 || rank > kMaxKt || rank > d->N) return fail(DMF_E_SHAPE, "resid: 1 <= rank <= min(N, 32) required");
    if (!Vh || !inv_sigma || !sums || (d->M && !U)) return fail(DMF_E_ARG, "NULL argument");
    CUDA_TRY(cudaSetDevice(h->device));
    cudaStream_t st = (cudaStream_t)stream;
    char* base = static_cast<char*>(ws);
    if (d->M == 0) {
        CUDA_TRY(cudaMemsetAsync(sums, 0, 2 * (size_t)rank * sizeof(double), st));
        return DMF_OK;
    }
    FitDev f;
    memset(&f, 0, sizeof(f));
    f.part = reinterpret_cast<double*>(base + p.off_ppart);
    f.gpart = reinterpret_cast<double*>(base + p.off_pgpart);
    f.tickets = reinterpret_cast<unsigned*>(base + p.off_ptickets);
    CUDA_TRY(cudaMemcpyAsync(base + p.off_pfit, &f, sizeof(f), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemsetAsync(base + p.off_ptickets, 0, p.off_ppart - p.off_ptickets, st));
    ProjArgs a;
    memset(&a, 0, sizeof(a));
    Geom& g = a.g;
    g.M = d->M; g.N = d->N; g.K = d->K;
    g.ldx = d->ldx; g.ldr = d->K ? d->ldr : 0;
    g.n_parts = p.p_parts; g.n_groups = p.p_groups; g.part_stride = 2 * kMaxKt;
    a.fit = reinterpret_cast<const FitDev*>(base + p.off_pfit);
    a.X = d->X; a.R = d->R; a.H1 = d->H1; a.Vh = Vh; a.inv_s = inv_sigma; a.U = U; a.sums = sums; a.rank = rank;
    resid_project_kernel<<<p.p_parts, kThreads, 0, st>>>(a);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaStreamSynchronize(st));                 // `f` is a stack temporary
    return DMF_OK;
}

int dmf_nndsvd_apply(const double* U, int64_t M, const double* Vh, const double* S, const double* sums, int32_t N, int32_t rank,
                     double* W, double* H, void* stream) {
    if (!Vh || !S || !sums || !H || M < 0 || N <= 0 || rank <= 0 || (M && (!U || !W))) return fail(DMF_E_ARG, "nndsvd: bad argument");
    const int blocks = (int)std::max<long long>(1, std::min<long long>((M + 255) / 256, 1024));
    nndsvd_apply_kernel<<<dim3(rank, blocks, 1), 256, 0, (cudaStream_t)stream>>>(U, M, Vh, S, sums, N, rank, W, H);
    CUDA_TRY(cudaGetLastError());
    return DMF_OK;
}

}  // extern "C"
