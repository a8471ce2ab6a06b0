// mg_step.cu — K1: MiniGridEnv.step (minigrid_env.py:525-595) fused with gen_obs (:597-650) and with the
// vector-level autoreset (MiniGridEnv.reset, :119-157) for a batch: ONE launch per vector step.
//
// One warp = one tile of 32 environments, one lane per environment.
//   1. lane 0 issues a TMA bulk copy (cp.async.bulk -> SASS UBLKCP) of the tile's interleaved grid words
//      into shared memory and arms an mbarrier with the byte count; meanwhile every lane loads its
//      action and 16-byte agent record with coalesced loads. Warps are persistent (one CTA per SM, one wave): one
//      buffer per warp, 22 warps at 72 registers (configure_step).
//   2. autoreset (NEXT_STEP: envs flagged last step, before the transition; SAME_STEP: envs that just ended,
//      after it): rare; the pending lanes replay their env's numpy-exact RNG draws while the idle lanes copy the level
//      template over those envs, then the warp patches the few draw-dependent cells (warp_reset).
//   3. transition: the 7-action rule on (agent, carrying, the one cell in front), predicated, with the
//      rare cell mutation written to the staged tile and straight back to HBM (2 byte stores).
//   4. observation in registers (mg_obs.cuh), staged into the consumed tile buffer in output layout, then one
//      TMA bulk store of the warp's 32 x 147 = 4704 contiguous bytes.
//   5. coalesced stores of direction / reward / terminated / truncated and the agent record.
// Large grids (LAYOUT_WINDOW) skip step 1: each lane gathers only the 7 lines its view needs straight into registers
// (21 independent 4-byte loads, one round trip; mg_obs.cuh: load_view_words), and the transition reads its front cell
// out of the same words. This file holds the tiled instantiations, mg_step_window.cu the window ones.
#include "mg_step_kernel.cuh"

namespace mg {

#ifdef MG_TIMELINE
int debug_timeline_window(void *out);
extern "C" int mg_debug_timeline(void *out, int layout) {  // out: unsigned long long[2][160][16]; layout: LAYOUT_* of the handle
  if (layout == LAYOUT_WINDOW) return debug_timeline_window(out);
  return (int)cudaMemcpyFromSymbol(out, g_tl, sizeof(g_tl));
}
#endif

static StepKernel step_kernel(int kind, int vis, int layout) {
  return layout == LAYOUT_WINDOW ? step_kernel_window(kind, vis) : pick_vis<LAYOUT_TILED>(kind, vis);
}

// Choose the CTA shape once per handle: one persistent CTA per SM. Measured on the final kernels
// (profiles/r02o..r02q_gpu_call.log, 262144 envs, desynchronised episodes): the tiled kernel at 72 registers wants about
// 22 warps (20..22 is a plateau, 24..28 a little behind, 16 clearly), the window kernel all 20 warps its 96 registers
// allow (at 72 registers and 28 warps it spills and loses), and the table-driven process_vis (32 KB of shared memory)
// beats the ALU form. MINIGRID_B200_CFG="warps" overrides the warp count (tuning and test knob).
cudaError_t configure_step(const Params &p, StepPlan *plan) {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int want_warps = 0;
  if (const char *cfg = getenv("MINIGRID_B200_CFG")) sscanf(cfg, "%d", &want_warps);
  const bool win = p.g.layout == LAYOUT_WINDOW;
  const int vis = p.see_through ? VIS_NONE : VIS_TBL;
  const int wcap = win ? 20 : 28;  // __launch_bounds__ of the kernel
  int wmax = wcap;  // the most warps whose buffers fit
  while (wmax >= 1 && step_smem_bytes(p.g, vis, wmax) > 227 * 1024 - 1024) --wmax;
  const int w = want_warps ? want_warps : min(win ? 20 : 22, wmax);
  if (w < 1 || w > wmax) return cudaErrorInvalidValue;
  StepKernel k = step_kernel(p.kind, vis, p.g.layout);
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)step_smem_bytes(p.g, vis, wmax));
  if (e != cudaSuccess) return e;
  const size_t smem = step_smem_bytes(p.g, vis, w);
  int ctas = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctas, k, w * 32, smem);
  if (e != cudaSuccess) return e;
  if (ctas * w > wcap) ctas = wcap / w;
  if (ctas < 1) return cudaErrorInvalidValue;
  plan->warps = w; plan->vis = vis; plan->ctas_per_sm = ctas; plan->smem = smem;
  const long long want = ((long long)p.n_tiles + plan->warps - 1) / plan->warps;
  long long grid = (long long)sms * plan->ctas_per_sm;
  if (grid > want) grid = want;
  // test knob: fewer CTAs than the device offers, so that a SMALL batch gives every warp several tiles (the tile loop's
  // prefetch / order list are otherwise only exercised at BASELINE sizes)
  if (const char *e = getenv("MINIGRID_B200_GRID")) { const long long cap = atoll(e); if (cap >= 1 && cap < grid) grid = cap; }
  plan->grid = (int)(grid < 1 ? 1 : grid);
  return cudaSuccess;
}

cudaError_t launch_step(const Params &p, const StepPlan &plan, const void *actions, int action_dtype, uint8_t *obs,
                        int32_t *dir, double *reward, uint8_t *term, uint8_t *trunc, uint32_t *packed, int step_parity,
                        cudaStream_t stream) {
  int tma_ok = ((reinterpret_cast<uintptr_t>(obs) & 15u) == 0) ? 1 : 0;
  tma_ok |= (step_parity & 1) << 2;  // direction of the unflagged tiles in K1's order list
#ifdef MG_TIMELINE
  static int launch_no = 0;
  tma_ok |= (launch_no++ & 1) << 1;
#endif
  StepKernel k = step_kernel(p.kind, plan.vis, p.g.layout);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)plan.grid);
  cfg.blockDim = dim3((unsigned)plan.warps * 32);
  cfg.dynamicSmemBytes = plan.smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, k, p, actions, action_dtype, obs, dir, reward, term, trunc, packed, tma_ok);
}

}  // namespace mg
