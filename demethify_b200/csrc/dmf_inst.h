// dmf_inst.h — kernel lookup functions, one set per (element type, weight storage) translation unit.
#pragma once
#include "dmf_device.cuh"
namespace dmf {
typedef void (*kern_t)(const PassArgs);
struct FusedArgs;
typedef void (*fused_kern_t)(const FusedArgs);
struct WlsArgs;
typedef void (*wls_kern_t)(const WlsArgs);
// Instantiated U-pass and rowgram kernels: known bucket, unknown bucket, columns per thread, rows per thread and tile.
// dmf_inst_body.cuh instantiates exactly these entries; make_plan takes the first entry whose buckets cover the shape.
struct KernEntry { int kb, nub, c, rpt; };
constexpr KernEntry kUTable[] = {{6, 2, 2, 4}, {8, 2, 2, 4}, {8, 8, 2, 1}, {16, 2, 2, 4}, {16, 8, 2, 1}, {16, 16, 1, 1},
                                 {32, 2, 1, 4}, {32, 8, 1, 1}, {32, 32, 1, 1}};
// c == 4 is rowgram4_kernel: rpt is its register rows, it walks 4 rows per thread and tile in batches of them
constexpr KernEntry kRowgramTable[] = {{0, 1, 4, 4},  {0, 2, 4, 4},  {0, 4, 4, 2},  {0, 8, 4, 1},  {6, 1, 4, 4},
                                       {6, 2, 4, 4},  {6, 4, 4, 2},  {6, 8, 4, 1},  {16, 1, 2, 4}, {16, 2, 2, 3},
                                       {16, 4, 2, 2}, {32, 1, 1, 4}, {32, 2, 1, 3}, {32, 4, 1, 2}};
#define DMF_DECL(TAG)                                      \
    kern_t pick_cost_##TAG(int ktb, int nub, int c);       \
    kern_t pick_alpha_##TAG(int ktb, int nub, int c);      \
    kern_t pick_u_##TAG(int kb, int nub, int);             \
    kern_t pick_rowgram_##TAG(int kb, int nub, int initial); \
    kern_t pick_panel_##TAG(int pb, int, int);             \
    kern_t pick_uinner_##TAG(int nub, int, int);           \
    kern_t pick_ainner_##TAG(int ktb, int, int);           \
    fused_kern_t pick_fused_##TAG(int kb, int nub, int s);   \
    wls_kern_t pick_wls_##TAG();
DMF_DECL(f64_f64) DMF_DECL(f64_u16) DMF_DECL(f32_f32) DMF_DECL(f32_u16)
#undef DMF_DECL
}  // namespace dmf
