// plan_probe.cu — host-only probe of the launch planner (make_plan in dmf_api.cu), built by tests/test_plan_cpu.py against the
// library's instantiation objects.  It makes no CUDA call: it reads one shape per stdin line
//   M N K n_u dtype wtype mode n_fits max_ctas_per_fit u_slots ldx ldd ldr ldu u_slot form      (form: 0 plain, 1 multiplicity, 2 gather)
// and prints one JSON object per line: the geometry of every engine the planner makes available, the kernels it would launch that
// resolve to nothing, the dispatch entries a fit on each engine launches ("launch") and the workspace regions.
//   plan_probe universe   prints every dispatch entry: a (lookup function, storage tag, arguments) triple over the domain of the
//                         kernel tables (dmf_inst_body.cuh) that resolves to a kernel, one name per line
//   plan_probe scan       prints the dispatch entries that some shape of the planner's whole domain launches on some engine
//                         (N 1..512, K + n_u <= 32, every storage tag, mode and form, three pitch styles), one name per line,
//                         then one line "combo <storage tag> <engine> <mode>" per combination some shape offers
#include <map>
#include <set>
#include <tuple>

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

// ---- dispatch entries.  The name holds every argument the lookup function reads, e.g. rowgram<f32_f32>[kb=16,nub=2,initial=1]
enum Fn { F_COST, F_ALPHA, F_U, F_ROWGRAM, F_PANEL, F_UINNER, F_AINNER, F_FUSED, F_WLS };
const char* const kTag[4] = {"f64_f64", "f64_u16", "f32_f32", "f32_u16"};   // the order of by_types
wls_kern_t (*const g_wls[4])() = {pick_wls_f64_f64, pick_wls_f64_u16, pick_wls_f32_f32, pick_wls_f32_u16};

std::vector<std::string> g_names;                               // entry id -> name
std::map<std::tuple<int, int, const void*>, int> g_entry;       // (function, tag, kernel) -> entry id

std::string entry_name(int fn, int tag, int a, int b, int c) {
    char buf[128];
    const char* t = kTag[tag];
    switch (fn) {
        case F_COST: snprintf(buf, sizeof buf, "cost<%s>[ktb=%d,c=%d,initial=%d]", t, a, c, b); break;
        case F_ALPHA: snprintf(buf, sizeof buf, "alpha<%s>[ktb=%d,c=%d]", t, a, c); break;
        case F_U: snprintf(buf, sizeof buf, "u<%s>[kb=%d,nub=%d]", t, a, b); break;
        case F_ROWGRAM: snprintf(buf, sizeof buf, "rowgram<%s>[kb=%d,nub=%d,initial=%d]", t, a, b, c); break;
        case F_PANEL: snprintf(buf, sizeof buf, "%s<%s>[pb=%d,c=%d]", c == 0 ? "panel" : (c == 1 ? "panel_mult" : "panel_mult_u1"), t, a, b); break;
        case F_UINNER: {
            const char* k[4] = {"u_inner", "u_inner_mult", "cost_cross", "usum"};
            snprintf(buf, sizeof buf, "%s<%s>[nub=%d]", k[b], t, a);
            break;
        }
        case F_AINNER: snprintf(buf, sizeof buf, "alpha_inner<%s>[ktb=%d]", t, a); break;
        case F_FUSED: snprintf(buf, sizeof buf, "fused<%s>[kb=%d,nub=%d,s=%d]", t, a, b, c); break;
        default: snprintf(buf, sizeof buf, "wls<%s>", t);
    }
    return buf;
}

void add_entry(int fn, int tag, int a, int b, int c, const void* k) {
    if (!k) return;
    const std::string name = entry_name(fn, tag, a, b, c);
    const auto key = std::make_tuple(fn, tag, k);
    const auto it = g_entry.find(key);
    if (it != g_entry.end()) {
        if (g_names[it->second] != name) {           // one kernel under two names: the name misses an argument the lookup reads
            fprintf(stderr, "plan_probe: %s and %s resolve to the same kernel\n", g_names[it->second].c_str(), name.c_str());
            exit(2);
        }
        return;
    }
    for (const std::string& n : g_names)
        if (n == name) {                               // one name, two kernels: the name ignores an argument the lookup reads
            fprintf(stderr, "plan_probe: %s resolves to two kernels\n", name.c_str());
            exit(2);
        }
    g_entry[key] = (int)g_names.size();
    g_names.push_back(name);
}

// every argument combination of the tables' domain (arguments beyond it select nothing or a duplicate)
void build_universe() {
    for (int t = 0; t < 4; ++t) {
        for (int a = 0; a <= 32; ++a) {
            for (int c = 0; c <= 4; ++c) {
                for (int b = 0; b <= 1; ++b) add_entry(F_COST, t, a, b, c, (const void*)g_cost[t](a, b, c));
                add_entry(F_ALPHA, t, a, 0, c, (const void*)g_alpha[t](a, 0, c));
                for (int m = 0; m <= 2; ++m) add_entry(F_PANEL, t, a, c, m, (const void*)g_panel[t](a, c, m));
            }
            for (int b = 0; b <= 32; ++b) {
                add_entry(F_U, t, a, b, 0, (const void*)g_u[t](a, b, 0));
                for (int c = 0; c <= 1; ++c) add_entry(F_ROWGRAM, t, a, b, c, (const void*)g_rowgram[t](a, b, c));
                for (int c = 0; c <= 4; ++c) add_entry(F_FUSED, t, a, b, c, (const void*)g_fused[t](a, b, c));
            }
            for (int w = 0; w <= 3; ++w) add_entry(F_UINNER, t, a, w, 0, (const void*)g_uinner[t](a, w, 0));
            add_entry(F_AINNER, t, a, 0, 0, (const void*)g_ainner[t](a, 0, 0));
        }
        add_entry(F_WLS, t, 0, 0, 0, (const void*)g_wls[t]());
    }
}

int tag_of(const dmf_shape_t& s) { return (s.dtype == DMF_F64 ? 0 : 2) + (s.wtype == DMF_W_U16 ? 1 : 0); }
int entry_of(int fn, const dmf_shape_t& s, const void* k) {
    const auto it = g_entry.find(std::make_tuple(fn, tag_of(s), k));
    return it == g_entry.end() ? -1 : it->second;
}

// The dispatch entries a dmf_fit_batched call launches on each engine the batch offers (-1: a launch that resolves to nothing).
// Stream: dmf_pass_init, dmf_pass_u, dmf_pass_alpha / dmf_pass_fw, dmf_pass_cost.  Gram: dmf_gram_init (rowgram, known-block
// panels) and dmf_gram_outer (u_inner, panels, alpha_inner, rowgram), with the multiplicity form's cost_cross and usum.  Fused:
// dmf_gram_init, dmf_fused_outer (fused pass, alpha_inner) and dmf_fused_finish (rowgram).
struct Launches { std::vector<int> e[3]; bool on[3]; };
Launches launches_of(dmf_batch_s* b) {
    const dmf_shape_t& s = b->shape;
    const Plan& q = b->p;
    Launches L{};
    L.on[0] = !b->multmode;
    if (L.on[0])
        L.e[0] = {entry_of(F_COST, s, (const void*)k_cost(b, 1)), entry_of(F_COST, s, (const void*)k_cost(b, 0)),
                  entry_of(F_U, s, (const void*)k_u(b)), entry_of(F_ALPHA, s, (const void*)k_alpha(b))};
    L.on[1] = q.gram_ok;
    if (L.on[1]) {
        std::vector<int>& g = L.e[1];
        g = {entry_of(F_ROWGRAM, s, (const void*)k_rowgram(b, 1)), entry_of(F_ROWGRAM, s, (const void*)k_rowgram(b, 0)),
             entry_of(F_UINNER, s, (const void*)k_uinner(b)), entry_of(F_AINNER, s, (const void*)k_ainner(b))};
        if (s.K) g.push_back(entry_of(F_PANEL, s, (const void*)k_panel(b)));
        g.push_back(entry_of(F_PANEL, s, (const void*)(b->multmode && s.n_u == 1 ? k_panel_u1(b) : k_panel(b))));
        if (b->multmode) {
            g.push_back(entry_of(F_UINNER, s, (const void*)k_costcross(b)));
            g.push_back(entry_of(F_UINNER, s, (const void*)k_usum(b)));
        }
    }
    L.on[2] = q.fused_ok;
    if (L.on[2]) {
        std::vector<int>& f = L.e[2];
        f = {entry_of(F_ROWGRAM, s, (const void*)k_rowgram(b, 1)), entry_of(F_ROWGRAM, s, (const void*)k_rowgram(b, 0)),
             entry_of(F_FUSED, s, (const void*)by_types_f(s, q.kb_f, q.nub_f, q.s_f)), entry_of(F_AINNER, s, (const void*)k_ainner(b))};
        if (s.K) f.push_back(entry_of(F_PANEL, s, (const void*)k_panel(b)));
    }
    return L;
}

// the batch-specific part of dmf_batch_create: gather form, multiplicity form, its one-unknown panel, the fused engine's exclusions
void batch_of(dmf_batch_s& b, const dmf_shape_t& s, const Plan& p, int form) {
    b.shape = s;
    b.p = p;
    b.multmode = form == 1;
    b.p.p1_ok = b.multmode && p.p1_ok;
    b.p.fused_ok = p.fused_ok && form == 0;
    if (b.multmode) std::copy(p.tx_mult, p.tx_mult + kMaxSrc, b.p.gg.tile_tx);
}

// the planner's whole domain: every shape it accepts, with DeviceProblem's pitches, the smallest even pitches and 16-byte pitches
int scan(const dmf_handle_s& h) {
    const char* const engine_names[3] = {"stream", "gram", "fused"};
    const char* const mode_names[3] = {"partial", "purity", "unsup"};      // DMF_MODE_*
    std::set<int> reached;
    std::set<std::string> combos;
    for (int tag = 0; tag < 4; ++tag)
        for (int K = 0; K < kMaxKt; ++K)
            for (int n_u = 1; K + n_u <= kMaxKt; ++n_u)
                for (int mode = 0; mode < 3; ++mode)
                    for (int N = 1; N <= 512; ++N)
                        for (int style = 0; style < 3; ++style)
                            for (int form = 0; form < 2; ++form) {
                                dmf_shape_t s{};
                                s.M = 100000; s.N = N; s.K = K; s.n_u = n_u;
                                s.dtype = tag < 2 ? DMF_F64 : DMF_F32; s.wtype = tag & 1 ? DMF_W_U16 : DMF_W_FLOAT;
                                s.mode = mode; s.n_fits = 1; s.u_slots = form == 1 ? 2 : 4;
                                const int es = s.dtype == DMF_F64 ? 8 : 4, ew = s.wtype == DMF_W_U16 ? 2 : es;
                                const auto even = [](long long v) { return v + (v & 1); };
                                const auto al16 = [](long long v, int e) { return (v * e + 15) / 16 * 16 / e; };
                                const bool wide = N * es >= 512;
                                const auto dev = [&](int e) { return wide ? ((N * e + 127) / 128 * 128 + 16) / e : (long long)(N + 7) / 8 * 8; };
                                if (style == 0) { s.ldx = dev(es); s.ldd = s.wtype == DMF_W_U16 ? dev(2) : s.ldx; }
                                else if (style == 1) { s.ldx = s.ldd = even(N); }
                                else { s.ldx = al16(even(N), es); s.ldd = al16(even(N), ew); }
                                s.ldr = even(K); s.ldu = even(n_u);
                                s.u_slot = al16(s.M * s.ldu, es);
                                Plan p;
                                if (make_plan(&h, s, p)) continue;
                                if (form == 1 && !p.mult_ok) continue;
                                dmf_batch_s b{};
                                batch_of(b, s, p, form);
                                const Launches L = launches_of(&b);
                                for (int e = 0; e < 3; ++e)
                                    if (L.on[e]) {
                                        reached.insert(L.e[e].begin(), L.e[e].end());
                                        combos.insert(std::string("combo ") + kTag[tag] + " " + engine_names[e] + " " + mode_names[mode]);
                                    }
                            }
    for (int id : reached)
        if (id >= 0) printf("%s\n", g_names[id].c_str());
    for (const std::string& c : combos) printf("%s\n", c.c_str());
    return 0;
}

}  // namespace

int main(int argc, char** argv) {
    const dmf_handle_s h{0, 148, 232448};
    build_universe();
    if (argc > 1 && !strcmp(argv[1], "universe")) {
        for (const std::string& n : g_names) printf("%s\n", n.c_str());
        return 0;
    }
    if (argc > 1 && !strcmp(argv[1], "scan")) return scan(h);
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
        dmf_batch_s b{};
        batch_of(b, s, p, form);
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

        const char* const engine_names[3] = {"stream", "gram", "fused"};
        const Launches L = launches_of(&b);
        printf(", \"launch\": {");
        for (int e = 0, first = 1; e < 3; ++e) {
            if (!L.on[e]) continue;
            printf("%s\"%s\": [", first ? "" : ", ", engine_names[e]);
            first = 0;
            for (size_t i = 0; i < L.e[e].size(); ++i) printf("%s\"%s\"", i ? ", " : "", L.e[e][i] < 0 ? "null" : g_names[L.e[e][i]].c_str());
            printf("]");
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
