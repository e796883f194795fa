// gx_fill_inst.cu -- instantiates gx_fill_kernel for one (K, CHAIN1) combination: compiled once per combination
// with -DGX_INST_K=4|8|16 -DGX_INST_CHAIN=0|1 (genomics_rs_b200/build.py builds the objects in parallel).
#include "gx_fill.cuh"

#if !defined(GX_INST_K) || !defined(GX_INST_CHAIN)
#error "compile with -DGX_INST_K=4|8|16 -DGX_INST_CHAIN=0|1"
#endif

namespace gx {

typedef void (*FillKernel)(const FillParams);

template <bool PROF>
static FillKernel pick_mode(bool L, bool C, int track, int band) {
    constexpr int K = GX_INST_K;
    constexpr bool CH = GX_INST_CHAIN != 0;
    if (band == BAND_DENSE) return gx_fill_kernel<K, false, true, 0, PROF, CH, BAND_DENSE>;   // global traceback with a code band
    // compact code storage.  Local: the start cell is already known (tile_best of the start-cell pass), no tracking
    if (band == BAND_COMPACT) return L ? gx_fill_kernel<K, true, true, 0, PROF, CH, BAND_COMPACT> : gx_fill_kernel<K, false, true, 0, PROF, CH, BAND_COMPACT>;
    if (track == 3) {   // first-maximum pass of GX_FLAG_LCS_AT_MAX: score only
        if (L) return gx_fill_kernel<K, true, false, 3, PROF, CH>;
        return gx_fill_kernel<K, false, false, 3, PROF, CH>;
    }
    if (!L && !C) return gx_fill_kernel<K, false, false, 0, PROF, CH>;
    if (!L && C) return gx_fill_kernel<K, false, true, 0, PROF, CH>;
    if (L && !C && track == 1) return gx_fill_kernel<K, true, false, 1, PROF, CH>;
    if (L && !C) return gx_fill_kernel<K, true, false, 2, PROF, CH>;
    return gx_fill_kernel<K, true, true, 2, PROF, CH>;
}

#define GX_CAT_(a, b, c, d) a##b##c##d
#define GX_CAT(a, b, c, d) GX_CAT_(a, b, c, d)
FillKernel GX_CAT(pick_fill_, GX_INST_K, _, GX_INST_CHAIN)(bool prof, bool L, bool C, int track, int band) {
    return prof ? pick_mode<true>(L, C, track, band) : pick_mode<false>(L, C, track, band);
}

}  // namespace gx
