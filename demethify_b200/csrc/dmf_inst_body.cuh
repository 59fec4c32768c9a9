// dmf_inst_body.cuh — included by dmf_inst_<tag>.cu with DMF_T, DMF_WT and DMF_TAG defined.
#include <iterator>
#include <utility>
#define DMF_INST_BODY
#include "dmf_inst.h"
#include "dmf_kernels.cuh"
#include "dmf_wls.cuh"
#include "dmf_gram.cuh"
#include "dmf_fused.cuh"
namespace dmf {
#define DMF_CAT2(a, b) a##b
#define DMF_CAT(a, b) DMF_CAT2(a, b)
// cost / set-up pass: (register-row bucket, columns per thread)
kern_t DMF_CAT(pick_cost_, DMF_TAG)(int ktb, int initial, int c) {
#define DMF_C(KTB_, C_)                                                                              \
    if (ktb == KTB_ && c == C_)                                                                      \
        return initial ? (kern_t)cost_kernel<DMF_T, DMF_WT, KTB_, C_, true> : (kern_t)cost_kernel<DMF_T, DMF_WT, KTB_, C_, false>;
    DMF_C(8, 2) DMF_C(16, 2) DMF_C(32, 1)
#undef DMF_C
    return nullptr;
}
kern_t DMF_CAT(pick_alpha_, DMF_TAG)(int ktb, int, int c) {
    if (ktb == 8 && c == 2) return alpha_pass_kernel<DMF_T, DMF_WT, 8, 2>;
    if (ktb == 16 && c == 2) return alpha_pass_kernel<DMF_T, DMF_WT, 16, 2>;
    if (ktb == 32 && c == 1) return alpha_pass_kernel<DMF_T, DMF_WT, 32, 1>;
    return nullptr;
}
// U pass and rowgram pass: the entries of kUTable / kRowgramTable (dmf_inst.h)
template <typename T, typename WT, size_t... I>
kern_t pick_u_in(int kb, int nub, std::index_sequence<I...>) {
    kern_t k = nullptr;
    ((kb == kUTable[I].kb && nub == kUTable[I].nub ? (void)(k = u_pass_kernel<T, WT, kUTable[I].kb, kUTable[I].nub, kUTable[I].c, kUTable[I].rpt>)
                                                   : (void)0), ...);
    return k;
}
kern_t DMF_CAT(pick_u_, DMF_TAG)(int kb, int nub, int) {
    return pick_u_in<DMF_T, DMF_WT>(kb, nub, std::make_index_sequence<std::size(kUTable)>());
}
template <typename T, typename WT, bool INITIAL, int I>
kern_t rowgram_at() {
    constexpr KernEntry e = kRowgramTable[I];
    if constexpr (e.c == 4) return rowgram4_kernel<T, WT, e.kb, e.nub, e.rpt, INITIAL>;
    else return rowgram_kernel<T, WT, e.kb, e.nub, e.c, e.rpt, INITIAL>;
}
template <typename T, typename WT, bool INITIAL, size_t... I>
kern_t pick_rowgram_in(int kb, int nub, std::index_sequence<I...>) {
    kern_t k = nullptr;
    ((kb == kRowgramTable[I].kb && nub == kRowgramTable[I].nub ? (void)(k = rowgram_at<T, WT, INITIAL, I>()) : (void)0), ...);
    return k;
}
kern_t DMF_CAT(pick_rowgram_, DMF_TAG)(int kb, int nub, int initial) {
    constexpr auto all = std::make_index_sequence<std::size(kRowgramTable)>();
    return initial ? pick_rowgram_in<DMF_T, DMF_WT, true>(kb, nub, all) : pick_rowgram_in<DMF_T, DMF_WT, false>(kb, nub, all);
}
// mult: 0 plain, 1 multiplicity form, 2 multiplicity form, u block of a single unknown type (PA = 1)
kern_t DMF_CAT(pick_panel_, DMF_TAG)(int pb, int c, int mult) {
    if (mult == 2) return (pb == 8 && c == 4) ? (kern_t)gram_panel_kernel<DMF_T, DMF_WT, 1, 8, 4, true> : nullptr;
    if (mult) return (pb == 8 && c == 4) ? (kern_t)gram_panel_kernel<DMF_T, DMF_WT, 2, 8, 4, true> : nullptr;
    if (pb == 8 && c == 4) return gram_panel_kernel<DMF_T, DMF_WT, 2, 8, 4, false>;
    if (pb == 16 && c == 1) return gram_panel_kernel<DMF_T, DMF_WT, 2, 16, 1, false>;
    return nullptr;
}
// which: 0 u_inner_kernel, 1 u_inner_mult_kernel, 2 cost_cross_kernel, 3 usum_kernel (the multiplicity form: nub <= 4)
kern_t DMF_CAT(pick_uinner_, DMF_TAG)(int nub, int which, int) {
#define DMF_UI(NUB_)                                                           \
    if (nub == NUB_) {                                                         \
        if (which == 0) return u_inner_kernel<DMF_T, NUB_>;                    \
        if (which == 1) return u_inner_mult_kernel<DMF_T, NUB_>;               \
        if (which == 3) return usum_kernel<DMF_T, NUB_>;                       \
        return cost_cross_kernel<DMF_T, NUB_>;                                 \
    }
    DMF_UI(1) DMF_UI(2) DMF_UI(4)
#undef DMF_UI
    return nub == 8 && which == 0 ? (kern_t)u_inner_kernel<DMF_T, 8> : nullptr;
}
kern_t DMF_CAT(pick_ainner_, DMF_TAG)(int ktb, int, int) {
    if (ktb == 8) return alpha_inner_kernel<DMF_T, 8>;
    if (ktb == 16) return alpha_inner_kernel<DMF_T, 16>;
    if (ktb == 32) return alpha_inner_kernel<DMF_T, 32>;
    return nullptr;
}
// fused engine (dmf_fused.cuh): FP64 storage only; (known bucket, unknown types, 8-sample blocks per warp)
template <typename T, typename WT>
struct FusedPick {
    static fused_kern_t get(int, int, int) { return nullptr; }
};
template <typename WT>
struct FusedPick<double, WT> {
    static fused_kern_t get(int kb, int nub, int s) {
#define DMF_F(KB_, NUB_, S_) \
    if (kb == KB_ && nub == NUB_ && s == S_) return fused_outer_kernel<WT, KB_, NUB_, S_>;
#define DMF_FS(KB_, NUB_) DMF_F(KB_, NUB_, 1) DMF_F(KB_, NUB_, 2) DMF_F(KB_, NUB_, 4)
        DMF_FS(0, 1) DMF_FS(0, 2) DMF_FS(4, 1) DMF_FS(4, 2) DMF_FS(6, 1) DMF_FS(6, 2) DMF_FS(8, 1) DMF_FS(8, 2)
#undef DMF_FS
#undef DMF_F
        return nullptr;
    }
};
fused_kern_t DMF_CAT(pick_fused_, DMF_TAG)(int kb, int nub, int s) { return FusedPick<DMF_T, DMF_WT>::get(kb, nub, s); }
wls_kern_t DMF_CAT(pick_wls_, DMF_TAG)() { return wls_moments_kernel<DMF_T, DMF_WT>; }
}  // namespace dmf
