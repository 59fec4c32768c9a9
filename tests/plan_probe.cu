// plan_probe.cu — host-only probe of the launch planner (make_plan in dmf_api.cu), built by tests/test_plan_cpu.py against the
// library's instantiation objects.  It makes no CUDA call: it reads one shape per stdin line
//   M N K n_u dtype wtype mode n_fits max_ctas_per_fit u_slots ldx ldd ldr ldu u_slot form      (form: 0 plain, 1 multiplicity, 2 gather)
// and prints one JSON object per line: the geometry of every engine the planner makes available, the kernels it would launch that
// resolve to nothing, and the workspace regions.
#include "dmf_api.cu"

namespace {

void print_list(const char* name, const unsigned* v, int n) {
    printf("\"%s\": [", name);
    for (int i = 0; i < n; ++i) printf("%s%u", i ? ", " : "", v[i]);
    printf("]");
}

void print_engine(const char* name, const Geom& g, unsigned smem, unsigned ring, bool first) {
    const unsigned off[kMaxSrc] = {g.offX, g.offD, g.offR, g.offU, g.offUp};
    printf("%s\"%s\": {\"ctas\": %d, \"groups\": %d, \"tile_rows\": %d, \"tiles\": %d, \"stages\": %d, \"stage_bytes\": %u, \"smem\": %u, \"ring\": %u, ",
           first ? "" : ", ", name, g.n_parts, g.n_groups, g.tile_rows, g.n_tiles, g.stages, g.stage_bytes, smem, ring);
    print_list("offs", off, kMaxSrc);
    printf(", ");
    print_list("tx", g.tile_tx, kMaxSrc);
    printf("}");
}

}  // namespace

int main() {
    const dmf_handle_s h{0, 148, 232448};
    dmf_shape_t s;
    int form;
    long long M, ldx, ldd, ldr, ldu, u_slot;
    while (scanf("%lld %d %d %d %d %d %d %d %d %d %lld %lld %lld %lld %lld %d", &M, &s.N, &s.K, &s.n_u, &s.dtype, &s.wtype, &s.mode, &s.n_fits,
                 &s.max_ctas_per_fit, &s.u_slots, &ldx, &ldd, &ldr, &ldu, &u_slot, &form) == 16) {
        s.M = M; s.ldx = ldx; s.ldd = ldd; s.ldr = ldr; s.ldu = ldu; s.u_slot = u_slot; s.reserved = 0;
        Plan p;
        const int rc = make_plan(&h, s, p);
        printf("{\"rc\": %d", rc);
        if (rc) {
            printf(", \"err\": \"%s\"}\n", g_err.c_str());
            continue;
        }
        if (form == 1 && !p.mult_ok) {      // dmf_batch_create rejects the batch
            printf(", \"mult_ok\": 0}\n");
            continue;
        }
        // the batch-specific part of dmf_batch_create: multiplicity form, its one-unknown panel, the fused engine's exclusions
        dmf_batch_s b{};
        b.shape = s;
        b.p = p;
        b.multmode = form == 1;
        b.p.p1_ok = b.multmode && p.p1_ok;
        b.p.fused_ok = p.fused_ok && form == 0;
        if (b.multmode) std::copy(p.tx_mult, p.tx_mult + kMaxSrc, b.p.gg.tile_tx);
        const Plan& q = b.p;
        printf(", \"mult_ok\": %d, \"cap\": %d, \"buckets\": {\"ktb\": %d, \"kb\": %d, \"nub\": %d, \"kb_g\": %d, \"nub_g\": %d, \"s_f\": %d}",
               p.mult_ok, h.max_smem_optin, p.ktb, p.kb, p.nub, p.kb_g, p.nub_g, p.s_f);

        std::vector<std::pair<const char*, kern_t>> launches = {
            {"cost", k_cost(&b, 0)}, {"cost_initial", k_cost(&b, 1)}, {"alpha", k_alpha(&b)}, {"u", k_u(&b)}};
        if (q.gram_ok) {
            launches.insert(launches.end(), {{"rowgram", k_rowgram(&b, 0)}, {"rowgram_initial", k_rowgram(&b, 1)}, {"panel", k_panel(&b)},
                                             {"u_inner", k_uinner(&b)}, {"alpha_inner", k_ainner(&b)}});
            if (b.multmode) launches.insert(launches.end(), {{"cost_cross", k_costcross(&b)}, {"usum", k_usum(&b)}, {"panel_u1", k_panel_u1(&b)}});
        }
        printf(", \"null_kernels\": [");
        int n_null = 0;
        for (const auto& l : launches)
            if (!l.second) printf("%s\"%s\"", n_null++ ? ", " : "", l.first);
        if (q.fused_ok && !by_types_f(s, q.kb_f, q.nub_f, q.s_f)) printf("%s\"fused\"", n_null++ ? ", " : "");
        printf("]");

        printf(", \"engines\": {");
        print_engine("stream", q.g, std::max({q.smem_cost, q.smem_alpha, q.smem_u}), kCtlBytes + kStages * q.g.stage_bytes, true);
        if (q.gram_ok) {
            print_engine("gram", q.gg, std::max(q.smem_rg, q.smem_panel), kCtlBytes + q.gg.stages * q.gg.stage_bytes, false);
            printf(", \"u_inner_ctas\": %d", q.n_parts_u);
        }
        if (q.p1_ok) print_engine("p1", q.gp1, q.smem_p1, kCtlBytes + q.gp1.stages * q.gp1.stage_bytes, false);
        if (q.fused_ok) {
            const FusedArgs& f = q.fa;
            const unsigned off[kMaxSrc] = {0, f.offD, f.offR, f.offU, f.offUp};
            printf(", \"fused\": {\"ctas\": %d, \"groups\": %d, \"tile_rows\": %d, \"tiles\": %d, \"stages\": %d, \"stage_bytes\": %u, \"smem\": %u, "
                   "\"ring\": %u, \"threads\": %d, \"stats\": %u, ",
                   f.g.n_parts, f.g.n_groups, q.fc.rows, f.n_tiles, q.fc.stages, f.stage_bytes, q.smem_f, kFusedCtlBytes + q.fc.stages * f.stage_bytes,
                   q.fc.threads, f.offStats);
            print_list("offs", off, kMaxSrc);
            printf("}");
        }
        printf("}");

        const size_t n = s.n_fits;
        const size_t regions[][2] = {{p.off_fits, sizeof(FitDev) * n}, {p.off_states, sizeof(FitState) * n}, {p.off_tickets, p.per_fit_tickets * n},
                                     {p.off_part, p.per_fit_part * n}, {p.off_gpart, p.per_fit_gpart * n}, {p.off_rowgram, p.per_fit_rowgram * n},
                                     {p.off_stats, p.per_fit_stats * n}, {p.off_gstats, p.per_fit_stats * n}, {p.off_red, p.per_fit_red * n},
                                     {p.off_usum, p.per_fit_usum * n}};
        printf(", \"ws_bytes\": %zu, \"ws\": [", p.ws_bytes);
        for (size_t i = 0; i < sizeof(regions) / sizeof(regions[0]); ++i) printf("%s[%zu, %zu]", i ? ", " : "", regions[i][0], regions[i][1]);
        printf("]}\n");
    }
    return 0;
}
