// d2d_tu_warp.cu - the instantiations of d2d_step_warp_kernel for ONE warps-per-block shape (-DD2D_TU_WPB=2 | 4 | 8; the
// library links three copies of this file, compiled in parallel).  Exports their entry points as the table
// d2d_warp_shape_<WPB> (d2d_internal.h).
#include "d2d_internal.h"
#include "d2d_step_warp.cuh"

#ifndef D2D_TU_WPB
#error "compile with -DD2D_TU_WPB=2, 4 or 8"
#endif
#define D2D_CAT2(a, b) a##b
#define D2D_CAT(a, b) D2D_CAT2(a, b)

namespace {
constexpr int WPB = D2D_TU_WPB;

// every instantiation d2d_step (plain or auto-reset) / d2d_step_many / d2d_episode may launch for this handle needs the dynamic shared-memory opt-in
template <bool PLE2, bool SPEC>
int allow_all(size_t smem) {
    int rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, false, SPEC, 0>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, true, SPEC, 0>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, true, WPB, false, SPEC, 0>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, true, WPB, true, SPEC, 0>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, false, SPEC, 1>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, true, WPB, false, SPEC, 1>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, false, SPEC, 2>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, true, SPEC, 3>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, true, SPEC, 4>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, false, SPEC, 5>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, false, WPB, true, SPEC, 5>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, true, WPB, false, SPEC, 5>, smem);
    if (!rc) rc = d2d_allow_smem(d2d_step_warp_kernel<PLE2, true, WPB, true, SPEC, 5>, smem);
    return rc;
}

size_t shape_smem(int R) { return d2d_warp_smem_bytes(R, WPB); }

template <bool PLE2, bool SPEC>
cudaError_t launch(const D2DParams &P, int grid, const D2DLaunchSel &sel, cudaStream_t st, bool pdl) {
#define D2D_GO(EXACT_, FULL_, MODE_) d2d_launch_step(d2d_step_warp_kernel<PLE2, EXACT_, WPB, FULL_, SPEC, MODE_>, grid, WPB * 32, shape_smem(P.R), st, P, pdl)
    // (an episode's drawn positions are exact in fp32, so it never needs the fp64 shadow path)
    if (sel.episode && sel.fast && sel.full) return sel.no_reset ? D2D_GO(false, true, 4) : D2D_GO(false, true, 3);
    if (sel.episode) return D2D_GO(false, false, 2);
    if (sel.many) return sel.exact ? D2D_GO(true, false, 1) : D2D_GO(false, false, 1);
    if (sel.autoreset) {
        if (sel.full) return sel.exact ? D2D_GO(true, true, 5) : D2D_GO(false, true, 5);
        return sel.exact ? D2D_GO(true, false, 5) : D2D_GO(false, false, 5);
    }
    if (sel.full) return sel.exact ? D2D_GO(true, true, 0) : D2D_GO(false, true, 0);
    return sel.exact ? D2D_GO(true, false, 0) : D2D_GO(false, false, 0);
#undef D2D_GO
}

int shape_plan(d2d_handle *h, size_t smem) {
    int rc;
    if (h->spec) {          // the reference's default EnvConfig shape: counts and division magics are immediates
        rc = allow_all<true, true>(smem);
        if (!rc) rc = d2d_plan_geometry(h, d2d_step_warp_kernel<true, false, WPB, true, true, 0>, WPB * 32, smem, WPB);
    } else if (h->ple2) {
        rc = allow_all<true, false>(smem);
        if (!rc) rc = d2d_plan_geometry(h, d2d_step_warp_kernel<true, false, WPB, true, false, 0>, WPB * 32, smem, WPB);
    } else {
        rc = allow_all<false, false>(smem);
        if (!rc) rc = d2d_plan_geometry(h, d2d_step_warp_kernel<false, false, WPB, true, false, 0>, WPB * 32, smem, WPB);
    }
    return rc;
}

cudaError_t shape_launch(const d2d_handle *h, const D2DParams &P, int grid, const D2DLaunchSel &sel, cudaStream_t st, bool pdl) {
    if (h->spec) return launch<true, true>(P, grid, sel, st, pdl);
    if (h->ple2) return launch<true, false>(P, grid, sel, st, pdl);
    return launch<false, false>(P, grid, sel, st, pdl);
}

// the fp64 pass reads 10^(p/10) from this translation unit's constant bank (per device: set at every d2d_create)
cudaError_t shape_tables(const double *pwr_lin_d) {
    return cudaMemcpyToSymbol(d2d_pwr_lin_c, pwr_lin_d, sizeof(double) * D2D_MAX_PWR_LEVELS);
}

#ifdef D2D_TIMELINE
// instrumented build (profiles/timeline.py): the stamp table is a __device__ variable of d2d_common.cuh, so every translation unit
// has its own copy - the one this shape's kernels write is read here
cudaError_t shape_timeline(void *host_out, size_t bytes) {
    return cudaMemcpyFromSymbol(host_out, d2d_tl_buf, bytes < sizeof(d2d_tl_buf) ? bytes : sizeof(d2d_tl_buf));
}
#else
constexpr cudaError_t (*shape_timeline)(void *, size_t) = nullptr;
#endif
}  // namespace

extern const D2DWarpShape D2D_CAT(d2d_warp_shape_, D2D_TU_WPB) = {WPB, shape_smem, shape_plan, shape_launch, shape_tables, shape_timeline};
