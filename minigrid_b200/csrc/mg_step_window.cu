// mg_step_window.cu — the LAYOUT_WINDOW instantiations of K1 (large grids), see mg_step_kernel.cuh.
#include "mg_step_kernel.cuh"

namespace mg {

StepKernel step_kernel_window(int kind, int vis) { return pick_vis<LAYOUT_WINDOW>(kind, vis); }

#ifdef MG_TIMELINE
int debug_timeline_window(void *out) { return (int)cudaMemcpyFromSymbol(out, g_tl, sizeof(g_tl)); }
#endif

}  // namespace mg
