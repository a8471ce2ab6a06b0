// mg_step_kernel.cuh — K1, the step kernel template (see mg_step.cu for the overview). It is instantiated in two
// translation units, mg_step.cu (tiled layout) and mg_step_window.cu (window layout): ptxas's code for the tiled
// kernels measurably depends on what else it compiles alongside them (profiles/README.md, r01 A/B runs).
#pragma once
#include <cstdio>
#include <cstdlib>

#include "mg_common.cuh"
#include "mg_levels.cuh"
#include "mg_obs.cuh"
#include "mg_pcg64.cuh"
#include "mg_transition.cuh"
#include "mg_postfilter.cuh"

namespace mg {

#ifdef MG_TIMELINE  // debug build only (scripts/timeline.py): per-CTA %globaltimer stamps of the last two launches
static __device__ unsigned long long g_tl[2][160][16];  // one per translation unit: mg_debug_timeline(layout) reads the right one
//  // 0-7: CTA stamps; 8: regenerating tiles, 9 / 10: longest regenerating / plain tile (ns), 11: end of the last regenerating tile, 12: its pull index, 13: list ready
__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define MG_TL(slot) do { if (threadIdx.x == 0) g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x][slot] = gtime(); } while (0)
#define MG_TL_EXIT() do { if ((threadIdx.x & 31) == 0) { const unsigned long long t_ = gtime(); \
    atomicMax(&g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x][6], t_); atomicMin(&g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x][7], t_); } } while (0)
#else
#define MG_TL(slot) do { } while (0)
#define MG_TL_EXIT() do { } while (0)
#endif

// per-warp buffer: holds the staged tile (or the 32 lanes' view windows), then, once the gather has consumed it,
// the warp's 4704-byte observation block in output layout.
__host__ __device__ inline uint32_t step_buf_bytes(const Geom &g) {
  uint32_t b = g.layout == LAYOUT_TILED ? (uint32_t)g.wpe * 128u : 0u;  // window layout: the view words live in registers
  if (b < (uint32_t)OBS_TILE_BYTES) b = OBS_TILE_BYTES;
  return (b + 127u) & ~127u;
}
// Tiles whose environments regenerate in this step (NEXT_STEP autoreset: the previous step flagged them) take twice as
// long as a plain tile (9 us against 4.7 us, profiles/r02c_timeline.txt: the numpy-exact draws are one lane's serial
// chain). Left where they are they end up in a CTA's last round every step and the whole grid waits for one warp, so
// each CTA visits them FIRST: the order of its (up to ORDER_CAP) tiles is a list in shared memory, flagged tiles in
// front. The list is built in the prologue, i.e. before griddepcontrol.wait, from flags the previous launch may still
// be writing: a stale flag only costs the tile its place in the order, never correctness.
constexpr int ORDER_CAP = 1024;
// [cell table 1 KB][visibility table 32 KB, VIS_TBL only][warps x buffer][warps x mbarrier][table mbarrier][tile counter][order list]
__host__ __device__ inline size_t step_smem_bytes(const Geom &g, int vis, int warps) {
  return 1024 + (vis == VIS_TBL ? VIS_TBL_BYTES : 0) + (size_t)warps * step_buf_bytes(g) + 8 * (size_t)warps + 32 + 2 * ORDER_CAP;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
               "l"(src), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tma_store_1d(void *dst, uint32_t src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(src), "r"(bytes) : "memory");
}

// volatile asm loads: they stay where they are written (ahead of the mbarrier wait), so a prefetch really is one
__device__ __forceinline__ uint4 ldg_rec(const uint4 *ptr) {
  uint4 v;
  asm volatile("ld.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(ptr));
  return v;
}
__device__ __forceinline__ void prefetch_rng(const RngRec *r) {  // 48 bytes: two 32-byte sectors
  asm volatile("prefetch.global.L2 [%0];" ::"l"(r));
  asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char *>(r) + 32));
}
__device__ __forceinline__ int load_action(const void *actions, int dtype, int env) {
  int v;
  if (dtype == 1) {
    long long w;
    asm volatile("ld.global.nc.s64 %0, [%1];" : "=l"(w) : "l"(reinterpret_cast<const long long *>(actions) + env));
    return (int)w;
  }
  if (dtype == 2) {
    asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(reinterpret_cast<const uint8_t *>(actions) + env));
    return v;
  }
  asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(v) : "l"(reinterpret_cast<const int *>(actions) + env));
  return v;
}

// OBJECT_TO_IDX type of a cell code (door states and the key-hiding box folded back)
__device__ __forceinline__ uint32_t code_type(uint32_t code) {
  const uint32_t t4 = code & 15u;
  return (t4 == T4_DOOR_CLOSED || t4 == T4_DOOR_LOCKED) ? (uint32_t)T_DOOR : (t4 == T4_BOX_WITH_KEY ? (uint32_t)T_BOX : t4);
}
// The reference's reward wrappers around one env's step, BonusWrapper(NoDeath(env)).step (wrappers.py:106-125, 163-184,
// 852-882). Out of line and behind one uniform branch: the hot loop must not carry their registers.
//   f0   the cell in front BEFORE the env stepped (Dynamic-Obstacles: before its balls moved), cur the cell under the agent after
struct WrapOut { double reward; uint32_t terminated; };
static __device__ __noinline__ WrapOut wrap_step(const Params &p, int env, bool active, int action_raw, uint32_t f0, uint32_t cur,
                                                 int ax, int ay, int dir, double reward, uint32_t terminated) {
  if (p.no_death_mask) {
    const bool going_to_death = action_raw == A_FORWARD && f0 != CODE_EMPTY && ((p.no_death_mask >> code_type(f0)) & 1);
    const bool in_death = cur != CODE_EMPTY && ((p.no_death_mask >> code_type(cur)) & 1);
    if (terminated && (going_to_death || in_death)) {
      terminated = 0u;
      reward = __dadd_rn(reward, p.death_cost);
    }
  }
  if (p.bonus_mode && active && (unsigned)action_raw <= (unsigned)A_DONE) {  // the state after the step keys the count
    uint32_t key = (uint32_t)(ay * p.g.W + ax);
    uint32_t per = (uint32_t)(p.g.W * p.g.H);
    if (p.bonus_mode == 1) { key = (key * 4u + (uint32_t)dir) * 7u + (uint32_t)action_raw; per *= 28u; }
    uint32_t *cnt = p.counts + (size_t)env * per + key;
    const uint32_t c = *cnt + 1u;
    *cnt = c;
    reward = __dadd_rn(reward, __ddiv_rn(1.0, __dsqrt_rn((double)c)));  // 1 / math.sqrt(new_count): both correctly rounded
  }
  WrapOut o = {reward, terminated};
  return o;
}

// MiniGridEnv.reset() for the lanes in `pend`. Phase 1: every pending lane replays the numpy-exact draws of ITS
// environment (lane per env; only the rejection loops diverge). Phase 2, one environment at a time with the whole
// warp: the owner's drawn integers are broadcast, lane L copies words L, L+32, ... of the level template into HBM
// (and into the staged tile when there is one), then the few cells that depend on the draw are re-evaluated and
// written as bytes. Out of line: it is the rare path and must not cost the hot loop registers.
struct ResetOut { int ax, ay, dir, tx, ty; uint32_t aux; };  // tx, ty, aux: post-filter targets (0 for the other kinds)

template <int KIND>
__device__ __noinline__ ResetOut warp_reset(const Params &p, unsigned pend, int tile, uint32_t *gtile, int lane) {
  const Geom &g = p.g;
  Level L = blank_level();
  // SAME_STEP: the lanes have just read (front cell) and possibly written (pickup / drop / toggle) their columns of the
  // staged tile, and other lanes are about to overwrite the pending envs' columns: the ballot that brought the warp
  // here synchronises the lanes but orders no memory
  __syncwarp();
  // pending envs per tile from which every pending lane fills its own env (a truncation wave) instead of the warp going
  // through them one at a time. 8: by chance (LavaCrossing: 0.85 % of the envs end per step) 4 of 32 happen once per
  // step somewhere in a 262144-env batch, and that one tile then cost 35 us and set the step time (profiles/r02d_gpu_call.log)
  constexpr int DENSE_RESET_MIN = 8;
  const bool dense = __popc(pend) >= DENSE_RESET_MIN;
  if ((pend >> lane) & 1u) {
    RngRec *rr = p.rng + (size_t)tile * TILE + lane;
    Pcg r = load_rng(rr);
    draw_level<KIND>(p, r, L);
    store_rng(rr, r);
    if (KIND == KIND_DYNOBS) {  // the obstacle list of the new episode
      uint32_t ex[4];
      dynobs_pack(L, ex);
      p.extra[(size_t)tile * TILE + lane] = make_uint4(ex[0], ex[1], ex[2], ex[3]);
    }
  } else if (!dense) {
    // Sparse case: the draws are one lane's serial chain of a few microseconds. The other lanes use that time (divergent
    // paths of a warp interleave where one stalls) to copy the level template over the pending envs, four independent
    // loads at a time.
    const unsigned idle = ~pend;
    const int n_idle = __popc(idle), rank = __popc(idle & ((1u << lane) - 1u));
    for (unsigned m = pend; m; m &= m - 1) {
      const int src = __ffs(m) - 1;
      uint32_t *genv = p.grid + grid_word(g, tile * TILE + src, 0);
      const int gs = g.layout == LAYOUT_TILED ? 32 : 1;  // stride of an env's consecutive words
      int w = rank;
      for (; w + 3 * n_idle < g.wpe; w += 4 * n_idle) {
        const uint32_t a = __ldg(p.tmpl + w), b = __ldg(p.tmpl + w + n_idle), c = __ldg(p.tmpl + w + 2 * n_idle), d = __ldg(p.tmpl + w + 3 * n_idle);
        if (gtile) { gtile[w * 32 + src] = a; gtile[(w + n_idle) * 32 + src] = b; gtile[(w + 2 * n_idle) * 32 + src] = c; gtile[(w + 3 * n_idle) * 32 + src] = d; }
        genv[(size_t)w * gs] = a; genv[(size_t)(w + n_idle) * gs] = b; genv[(size_t)(w + 2 * n_idle) * gs] = c; genv[(size_t)(w + 3 * n_idle) * gs] = d;
      }
      for (; w < g.wpe; w += n_idle) {
        const uint32_t a = __ldg(p.tmpl + w);
        if (gtile) gtile[w * 32 + src] = a;
        genv[(size_t)w * gs] = a;
      }
    }
  }
  constexpr bool PF = has_post_filter<KIND>();
  const ResetOut out = {L.ax, L.ay, L.adir, PF ? level_tx(L) : 0, PF ? level_ty(L) : 0, PF ? level_aux(L) : 0u};
  __syncwarp();
  uint8_t *sb = reinterpret_cast<uint8_t *>(gtile), *gb = reinterpret_cast<uint8_t *>(p.grid);
  // Dense case (a synchronised truncation wave: under random actions nearly every env of a batch truncates in the
  // same step): every pending lane fills ITS OWN env — template words (one broadcast load per word; in the tiled
  // layout the 32 lanes' stores of a word index are one 128-byte line), then all patch cells of its own level —
  // instead of the warp going through the environments one at a time.
  if (dense) {
    if ((pend >> lane) & 1u) {
      const int env = tile * TILE + lane;
      for (int w = 0; w < g.wpe; ++w) {
        const uint32_t word = __ldg(p.tmpl + w);
        if (gtile) gtile[w * 32 + lane] = word;
        p.grid[grid_word(g, env, w)] = word;
      }
      for (int share = 0; share < 32; ++share)  // patch_level hands out the cells in 32 shares: take them all
        patch_level<KIND>(p, L, share, [&](int x, int y) {
          const uint8_t code = (uint8_t)cell_of<KIND>(p, L, x, y);
          const int rw = r_word(g, x, y), cw = c_word(g, x, y);
          if (gtile) { sb[((size_t)rw * 32 + lane) * 4 + (x & 3)] = code; sb[((size_t)cw * 32 + lane) * 4 + (y & 3)] = code; }
          gb[grid_word(g, env, rw) * 4 + (x & 3)] = code;
          gb[grid_word(g, env, cw) * 4 + (y & 3)] = code;
        });
    }
    __syncwarp();
    return out;
  }
  while (pend) {
    const int src = __ffs(pend) - 1;
    pend &= pend - 1;
    const int env = tile * TILE + src;
    Level B;  // the owner's draw, broadcast
    B.ax = B.ay = B.adir = 0;
    B.a = __shfl_sync(0xFFFFFFFFu, L.a, src); B.b = __shfl_sync(0xFFFFFFFFu, L.b, src);
    B.c = __shfl_sync(0xFFFFFFFFu, L.c, src); B.d = __shfl_sync(0xFFFFFFFFu, L.d, src);
    B.e = __shfl_sync(0xFFFFFFFFu, L.e, src); B.f = __shfl_sync(0xFFFFFFFFu, L.f, src);
    B.rv = __shfl_sync(0xFFFFFFFFu, L.rv, src); B.rh = __shfl_sync(0xFFFFFFFFu, L.rh, src);
    B.ov = __shfl_sync(0xFFFFFFFFu, L.ov, src); B.oh = __shfl_sync(0xFFFFFFFFu, L.oh, src);
    if (KIND == KIND_MULTIROOM || KIND == KIND_PLAYGROUND || KIND == KIND_GOTOOBJECT || KIND == KIND_FETCH || KIND == KIND_PUTNEAR || KIND == KIND_DYNOBS ||
        KIND == KIND_ROOMGRID) {
      const unsigned long long lo = __shfl_sync(0xFFFFFFFFu, (unsigned long long)L.rm03, src);
      const unsigned long long hi = __shfl_sync(0xFFFFFFFFu, (unsigned long long)(L.rm03 >> 64), src);
      B.rm03 = ((u128)hi << 64) | lo;
      B.rm45 = __shfl_sync(0xFFFFFFFFu, L.rm45, src);
      B.nrooms = __shfl_sync(0xFFFFFFFFu, L.nrooms, src);
    } else { B.rm03 = 0; B.rm45 = 0; B.nrooms = 0; }
    if (KIND == KIND_ROOMGRID) {
      const unsigned long long lo = __shfl_sync(0xFFFFFFFFu, (unsigned long long)L.rmx, src);
      const unsigned long long hi = __shfl_sync(0xFFFFFFFFu, (unsigned long long)(L.rmx >> 64), src);
      B.rmx = ((u128)hi << 64) | lo;
    } else B.rmx = 0;
    // (the template words were written by the idle lanes during the draws, ordered before this point by __syncwarp)
    patch_level<KIND>(p, B, lane, [&](int x, int y) {
      const uint8_t code = (uint8_t)cell_of<KIND>(p, B, x, y);
      const int rw = r_word(g, x, y), cw = c_word(g, x, y);
      if (gtile) { sb[((size_t)rw * 32 + src) * 4 + (x & 3)] = code; sb[((size_t)cw * 32 + src) * 4 + (y & 3)] = code; }
      gb[grid_word(g, env, rw) * 4 + (x & 3)] = code;
      gb[grid_word(g, env, cw) * 4 + (y & 3)] = code;
    });
  }
  __syncwarp();
  return out;
}

// LAYOUT_TILED: each warp stages its tile in one shared-memory buffer by a bulk copy. LAYOUT_WINDOW: each lane loads
// its view window into registers, and the warp fetches the next tile's agent records and actions one tile ahead.
template <int KIND, int VIS, int LAYOUT>
__global__ void __launch_bounds__(LAYOUT == LAYOUT_TILED ? 896 : 640, 1)  // one CTA per SM: tiled <= 28 warps (72 regs: 7 warps per scheduler), window <= 20 (96 regs: it keeps 21 view words live)
k_step(const __grid_constant__ Params p, const void *__restrict__ actions, int act_dtype, uint8_t *__restrict__ obs,
       int32_t *__restrict__ dir_out, double *__restrict__ reward_out, uint8_t *__restrict__ term_out,
       uint8_t *__restrict__ trunc_out, uint32_t *__restrict__ packed_out, int obs_tma_ok) {
  constexpr bool WIN = (LAYOUT == LAYOUT_WINDOW);  // agent records / actions / tile index are fetched one tile ahead
  extern __shared__ __align__(128) uint8_t smem_raw[];
  Geom g = p.g;
  g.layout = LAYOUT;  // both are implied by LAYOUT: let the compiler fold them
  g.ring = WIN ? 3 : 1;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int WARPS = blockDim.x >> 5;
  const uint32_t tile_bytes = (uint32_t)g.wpe * 128u;
  const uint32_t buf_bytes = step_buf_bytes(g);
  constexpr uint32_t TBL = (VIS == VIS_TBL) ? (uint32_t)VIS_TBL_BYTES : 0u;

  uint32_t *lut = reinterpret_cast<uint32_t *>(smem_raw);
  const uint16_t *vis_tbl = reinterpret_cast<const uint16_t *>(smem_raw + 1024);
  uint32_t *gtile = reinterpret_cast<uint32_t *>(smem_raw + 1024 + TBL + (size_t)warp * buf_bytes);
  uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw + 1024 + TBL + (size_t)WARPS * buf_bytes);
  const uint32_t bar = smem_u32(bars + warp), tbl_bar = smem_u32(bars + WARPS);
  int *s_next = reinterpret_cast<int *>(bars + WARPS + 1);
  uint16_t *s_order = reinterpret_cast<uint16_t *>(bars + WARPS + 3);

  // Programmatic dependent launch: let the next kernel in the stream start its prologue while this grid drains,
  // and do our own prologue (nothing the previous step wrote is touched) before waiting for it to complete.
  asm volatile("griddepcontrol.launch_dependents;");
#ifdef MG_TIMELINE
  if (threadIdx.x == 0) {
    g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x][6] = 0ull; g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x][7] = ~0ull;
    for (int i = 8; i < 16; ++i) g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x][i] = 0ull;
  }
#endif
  MG_TL(0);
  const bool stepping = actions != nullptr;  // nullptr: observation-only pass (MiniGridEnv.gen_obs), state untouched
  // one wave of persistent CTAs; CTA c owns tiles [c T/G, (c+1) T/G), its warps pull from a shared counter
  // (the first n_tiles % gridDim CTAs own one tile more; 32-bit arithmetic: no division subroutine in the prologue)
  const unsigned tq = (unsigned)p.n_tiles / gridDim.x, tr = (unsigned)p.n_tiles % gridDim.x;
  const int t_lo = (int)(blockIdx.x * tq + min(blockIdx.x, tr));
  const int t_hi = t_lo + (int)tq + (blockIdx.x < tr ? 1 : 0);
  // pull index k of a CTA: its k-th tile. k < WARPS: the static first round; behind it, the order list (flagged tiles first)
  const int n_my = t_hi - t_lo;
  const int m_ord = min(n_my, ORDER_CAP);
  const bool use_order = stepping && p.mode == AUTORESET_NEXT_STEP && m_ord > WARPS;
  if (threadIdx.x == 0) {
    *s_next = (WIN ? 2 : 1) * WARPS;
    if (VIS == VIS_TBL) {  // the table is immutable after mg_create: its copy may run ahead of griddepcontrol.wait
      mbar_init(tbl_bar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      mbar_expect_tx(tbl_bar, TBL);
      tma_load_1d(smem_u32(vis_tbl), p.vis_tbl, TBL, tbl_bar);
    }
  }
  auto map_tile = [&](int k) -> int {  // the CTA's k-th tile
    if (k >= n_my) return p.n_tiles;
    return t_lo + ((use_order && k < m_ord) ? (int)s_order[k] : k);
  };
  if (use_order && warp == WARPS - 1) {
    // tiles 0 .. m_ord - 1 of this CTA, those flagged by the previous step first. Ballots are kept in registers (lane c:
    // chunk c) so that both passes see the same flags whatever is written to them meanwhile.
    const uint8_t *hot = p.tile_hot + t_lo;
    unsigned mybal = 0;
    const int chunks = (m_ord + 31) >> 5;
    for (int c = 0; c < chunks; ++c) {
      const int idx = 32 * c + lane;
      uint32_t f = 0;
      if (idx < m_ord) asm volatile("ld.global.relaxed.gpu.u8 %0, [%1];" : "=r"(f) : "l"(hot + idx));
      const unsigned bal = __ballot_sync(0xFFFFFFFFu, f != 0);
      if (lane == c) mybal = bal;
    }
    int pre = __popc(mybal);  // inclusive scan over lanes of the chunks' hot counts
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xFFFFFFFFu, pre, d);
      if (lane >= d) pre += v;
    }
    const int hot_total = __shfl_sync(0xFFFFFFFFu, pre, 31);
    const int excl = pre - __popc(mybal);
    for (int c = 0; c < chunks; ++c) {
      const unsigned bal = __shfl_sync(0xFFFFFFFFu, mybal, c);
      const int hb = __shfl_sync(0xFFFFFFFFu, excl, c);
      const int idx = 32 * c + lane;
      if (idx < m_ord) {
        const unsigned lt = (1u << lane) - 1u;
        const bool is_hot = (bal >> lane) & 1u;
        // the unflagged tiles alternate their direction from step to step (bit 2 of obs_tma_ok): the tiles a CTA finished
        // last in the previous step are the ones whose flags this prologue may have read too early, and they come first now
        const int cold_rank = (32 * c - hb) + __popc(~bal & lt);
        const int pos = is_hot ? hb + __popc(bal & lt) : hot_total + ((obs_tma_ok & 4) ? (m_ord - hot_total - 1 - cold_rank) : cold_rank);
        s_order[pos] = (uint16_t)idx;
      }
    }
  }
  if (lane == 0) {
    mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  // the 256-entry (type, colour, state) table is pure arithmetic: no global load anywhere near the critical path
  for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = decode_cell((uint32_t)i);
  __syncthreads();
  MG_TL(1);
  asm volatile("griddepcontrol.wait;" ::: "memory");  // everything below reads state the previous step wrote
  MG_TL(2);
  bool first = true;  // first tile of this warp
  int tile = map_tile(warp);
  int next = WIN ? map_tile(WARPS + warp) : p.n_tiles;

  uint4 rec = make_uint4(0, 0, 0, 0);
  int action = A_DONE;
  if (WIN && tile < p.n_tiles) {
    const int env0 = tile * TILE + lane;
    rec = ldg_rec(p.agent + env0);
    if (stepping && env0 < p.n_envs) action = load_action(actions, act_dtype, env0);
    // an env that regenerates in this step starts from its RNG record: bring it in early
    if (stepping && ((rec.y >> 8) & FLAG_PENDING)) prefetch_rng(p.rng + env0);
  }

  uint8_t *gb = reinterpret_cast<uint8_t *>(p.grid);
  uint32_t phase = 0;  // parity to wait for on the warp's mbarrier
  while (tile < p.n_tiles) {
    uint4 rec_n = make_uint4(0, 0, 0, 0);
    int action_n = A_DONE, nn = p.n_tiles;
    if (WIN) {
      if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the previous obs block has left
      if (next < p.n_tiles) {  // the next tile's agent records and actions, and the index of the tile after it
        if (lane == 0) nn = map_tile(atomicAdd(s_next, 1));  // shared-memory atomic, consumed one tile later
        const int env_n = next * TILE + lane;
        rec_n = ldg_rec(p.agent + env_n);
        if (stepping && env_n < p.n_envs) action_n = load_action(actions, act_dtype, env_n);
      }
    } else {
      if (lane == 0) {
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");  // the previous obs block has left the buffer
        mbar_expect_tx(bar, tile_bytes);
        tma_load_1d(smem_u32(gtile), p.grid + (size_t)tile * g.wpe * 32, tile_bytes, bar);
      }
      const int env0 = tile * TILE + lane;
      rec = ldg_rec(p.agent + env0);
      action = (stepping && env0 < p.n_envs) ? load_action(actions, act_dtype, env0) : A_DONE;
      if (stepping && ((rec.y >> 8) & FLAG_PENDING)) prefetch_rng(p.rng + env0);
      // (Pulling the next tile's index here and asking L2 for its block a tile ahead was measured and rejected: DoorKey
      // 18.8 -> 20.2 us, Fetch 30.5 -> 34.1: committing a warp to its next tile one tile early costs more balance than
      // the shorter copy wins, profiles/r02w_gpu_call.log.)
    }
#ifdef MG_TIMELINE
    const unsigned long long tl_t0 = gtime();
    bool tl_hot = false;
#endif
    const int env = tile * TILE + lane;
    const bool active = env < p.n_envs;
    int ax = rec.x & 0xFF, ay = (rec.x >> 8) & 0xFF;
    int dir = rec.y & 3;
    uint32_t flags = rec.y >> 8;
    uint32_t carry = rec.z;
    int steps = (int)rec.w;
    constexpr bool PF = has_post_filter<KIND>();  // the record's spare bits hold the filter's targets
    int tx = PF ? (int)((rec.x >> 16) & 0xFFu) : 0, ty = PF ? (int)(rec.x >> 24) : 0;

    if (!WIN) {
      mbar_wait(bar, phase);
      phase ^= 1u;
#ifdef MG_TIMELINE
      if (first) MG_TL(3);
#endif
    } else {
      __syncwarp();  // lane 0 has waited for the bulk store that was still reading this buffer
    }

    const uint32_t *base = gtile + lane;
    double reward = 0.0;
    uint32_t terminated = 0, truncated = 0;
    int rsteps = 0;  // the step count the reward was computed from (a SAME_STEP autoreset zeroes `steps` afterwards)
    // NEXT_STEP autoreset (gymnasium >= 1.0 SyncVectorEnv): an env that ended last step ignores its action,
    // is reset now, and returns the reset obs with reward 0 / False / False
    bool fresh = false;
    bool wrote = false;  // this warp wrote grid bytes through the generic proxy during this tile
    if (stepping && p.mode == AUTORESET_NEXT_STEP) {
      fresh = active && (flags & FLAG_PENDING);
      const unsigned pend = __ballot_sync(0xFFFFFFFFu, fresh);
      if (pend) {
        wrote = true;
#ifdef MG_TIMELINE
        tl_hot = true;
#endif
        const ResetOut ro = warp_reset<KIND>(p, pend, tile, WIN ? nullptr : gtile, lane);
        if (fresh) {
          ax = ro.ax; ay = ro.ay; dir = ro.dir; carry = 0; steps = 0; flags &= ~FLAG_PENDING;
          if (PF) { tx = ro.tx; ty = ro.ty; flags = (flags & 0xFFu) | (ro.aux << 8); }
        }
      }
    }
    // LAYOUT_WINDOW: the view's words go straight to registers (mg_obs.cuh: load_view_words): 21 independent loads,
    // one memory round trip per step; the transition reads its front cell out of the same words.
    ViewWords vw;
    const uint32_t *envw = p.grid + (size_t)env * g.wpe;
    auto ldw = [&](int w) {
      uint32_t v;
      asm volatile("ld.global.u32 %0, [%1];" : "=r"(v) : "l"(envw + w));  // plain (coherent) load: this warp may just have regenerated the env
      return v;
    };
    if (WIN) {
      int dirn = dir;
      if (stepping && !fresh) dirn = (dir + (action == A_LEFT ? 3 : 0) + (action == A_RIGHT ? 1 : 0)) & 3;
      load_view_words(g, ax, ay, dirn, vw, ldw);
    }
    if (stepping && !fresh) {
      // ---- MiniGridEnv.step, minigrid_env.py:525-588 ----
      steps += 1;
      const int action_raw = action;  // what the wrappers saw (Dynamic-Obstacles remaps it below)
      int fx, fy;
      front_pos(g, ax, ay, dir, fx, fy);
      const int rw = r_word(g, fx, fy), cw = c_word(g, fx, fy);
      bool not_clear = false;
      uint32_t fc_before = 0;  // Dynamic-Obstacles: the front cell before the obstacles moved
      if (KIND == KIND_DYNOBS && !WIN) {
        // DynamicObstaclesEnv.step (dynamicobstacles.py:135-158): actions beyond forward count as left, the front cell is
        // looked at BEFORE the obstacles move, then every obstacle is re-placed with draws from the env's own stream
        if (action >= 3) action = A_LEFT;
        const uint32_t fc0 = (tile_word<true>(base, rw) >> (8 * (fx & 3))) & 0xFFu;
        not_clear = fc0 != CODE_EMPTY && (fc0 & 15u) != T_GOAL;
        fc_before = fc0;
        if (active) {
          RngRec *rr = p.rng + env;
          Pcg r = load_rng(rr);
          const uint4 e4 = p.extra[env];
          uint32_t ex[4] = {e4.x, e4.y, e4.z, e4.w};
          uint8_t *sb = reinterpret_cast<uint8_t *>(gtile);
          uint8_t *tb = reinterpret_cast<uint8_t *>(p.grid + (size_t)tile * g.wpe * 32);
          dynobs_move(g, r, p.kp[0], ex, ax, ay,
                      [&](int x, int y) { return (tile_word<true>(base, r_word(g, x, y)) >> (8 * (x & 3))) & 0xFFu; },
                      [&](int x, int y, uint32_t code) {
                        const int o_r = (r_word(g, x, y) * 32 + lane) * 4 + (x & 3), o_c = (c_word(g, x, y) * 32 + lane) * 4 + (y & 3);
                        sb[o_r] = (uint8_t)code; sb[o_c] = (uint8_t)code;
                        tb[o_r] = (uint8_t)code; tb[o_c] = (uint8_t)code;
                      });
          store_rng(rr, r);
          p.extra[env] = make_uint4(ex[0], ex[1], ex[2], ex[3]);
          wrote = true;
        }
      }
      uint32_t fc;
      const int fpos = ((dir & 1) ? ay : ax) + ((dir < 2) ? 1 : -1);  // the front cell's position on the agent's own line
      if (WIN) fc = view_words_byte(vw, fpos);  // meaningless after a turn (other array loaded), and then unused
      else fc = (tile_word<true>(base, rw) >> (8 * (fx & 3))) & 0xFFu;

      const uint32_t carry_before = carry;
      const int act = pre_filter<KIND>(action);
      const StepOut so = transition(act, fc, fx, fy, ax, ay, dir, carry);
      const uint32_t newc = so.newc;
      terminated = so.terminated;
      if (so.goal)  // _reward(), minigrid_env.py:240-245: host-computed table, never an FMA
        reward = steps <= p.max_steps ? p.reward_lut[steps]
                                      : __dsub_rn(1.0, __dmul_rn(0.9, __ddiv_rn((double)steps, (double)p.max_steps)));
      if (so.bad_action) atomicOr(p.err, ERR_BAD_ACTION);  // ValueError("Unknown action"), minigrid_env.py:584-585
      if (newc != fc && active) {
        wrote = true;
        if (!WIN) {
          uint8_t *sb = reinterpret_cast<uint8_t *>(gtile);
          sb[(rw * 32 + lane) * 4 + (fx & 3)] = (uint8_t)newc;
          sb[(cw * 32 + lane) * 4 + (fy & 3)] = (uint8_t)newc;
        } else {  // pickup / drop / toggle do not turn: the front cell is on the loaded centre line
          view_words_set_byte(vw, fpos, newc);
        }
        if (!WIN) {  // tile-relative addressing: 32-bit index math on the common path
          uint8_t *tb = reinterpret_cast<uint8_t *>(p.grid + (size_t)tile * g.wpe * 32);
          tb[(rw * 32 + lane) * 4 + (fx & 3)] = (uint8_t)newc;
          tb[(cw * 32 + lane) * 4 + (fy & 3)] = (uint8_t)newc;
        } else {
          gb[grid_word(g, env, rw) * 4 + (fx & 3)] = (uint8_t)newc;
          gb[grid_word(g, env, cw) * 4 + (fy & 3)] = (uint8_t)newc;
        }
      }
      if (KIND == KIND_DYNOBS && action == A_FORWARD && not_clear) {  // walked into an obstacle or a wall: :161-165
        reward = -1.0;
        terminated = 1u;
      }
      if (PF) {  // the env's own step(): a few predicates on top of MiniGridEnv.step (mg_postfilter.cuh)
        PostIn in;
        in.action = act; in.ax = ax; in.ay = ay; in.dir = dir;
        in.carry_before = carry_before; in.carry = carry;
        in.tx = tx; in.ty = ty; in.aux = flags >> 8;
        in.red_before = in.blue_before = in.red_after = in.blue_after = false;
        in.variant = p.kp[0]; in.door_open = false;
        if (KIND == KIND_ROOMGRID && p.kp[0] == RG_UNLOCK) {  // self.door.is_open: the cell at the target, after this step's mutation
          uint32_t cd;
          if (!WIN) cd = (tile_word<true>(base, r_word(g, tx, ty)) >> (8 * (tx & 3))) & 0xFFu;
          else cd = gb[grid_word(g, env, r_word(g, tx, ty)) * 4 + (tx & 3)];
          in.door_open = (cd & 15u) == T_DOOR;
        }
        if (KIND == KIND_REDBLUEDOORS) {  // a door changes only as the front cell of a toggle
          const int xl = g.H / 2, xr = g.H / 2 + g.H - 1;
          uint32_t cr, cb;
          if (!WIN) {
            cr = (tile_word<true>(base, r_word(g, xl, tx)) >> (8 * (xl & 3))) & 0xFFu;
            cb = (tile_word<true>(base, r_word(g, xr, ty)) >> (8 * (xr & 3))) & 0xFFu;
          } else {
            cr = gb[grid_word(g, env, r_word(g, xl, tx)) * 4 + (xl & 3)];
            cb = gb[grid_word(g, env, r_word(g, xr, ty)) * 4 + (xr & 3)];
          }
          in.red_after = (cr & 15u) == T_DOOR;
          in.blue_after = (cb & 15u) == T_DOOR;
          in.red_before = (fx == xl && fy == tx) ? (fc & 15u) == T_DOOR : in.red_after;
          in.blue_before = (fx == xr && fy == ty) ? (fc & 15u) == T_DOOR : in.blue_after;
        }
        const PostOut po = post_filter<KIND>(in, terminated);
        terminated = po.terminated;
        if (po.reward == POST_ZERO) reward = 0.0;
        if (po.reward == POST_REWARD)
          reward = steps <= p.max_steps ? p.reward_lut[steps]
                                        : __dsub_rn(1.0, __dmul_rn(0.9, __ddiv_rn((double)steps, (double)p.max_steps)));
      }
      if (p.no_death_mask | p.bonus_mode) {  // the reference's reward wrappers: rare, one uniform branch, out of line
        uint32_t cur = 0;  // the cell under the agent after the step
        if (p.no_death_mask) {
          if (WIN) cur = view_words_byte(vw, (dir & 1) ? ay : ax);
          else cur = (tile_word<true>(base, r_word(g, ax, ay)) >> (8 * (ax & 3))) & 0xFFu;
        }
        const WrapOut wo = wrap_step(p, env, active, action_raw, (KIND == KIND_DYNOBS && !WIN) ? fc_before : fc, cur, ax, ay, dir, reward, terminated);
        reward = wo.reward;
        terminated = wo.terminated;
      }
      truncated = steps >= p.max_steps;
      rsteps = steps;
      const bool done = (terminated | truncated) != 0;
      if (p.mode == AUTORESET_NEXT_STEP) flags = done ? (flags | FLAG_PENDING) : (flags & ~FLAG_PENDING);
    }
    // SAME_STEP autoreset: the env is reset inside the step that ended it and the reset obs is returned
    if (stepping && p.mode == AUTORESET_SAME_STEP) {
      const bool again = active && ((terminated | truncated) != 0);
      const unsigned pend = __ballot_sync(0xFFFFFFFFu, again);
      if (pend) {
        wrote = true;
        const ResetOut ro = warp_reset<KIND>(p, pend, tile, WIN ? nullptr : gtile, lane);
        if (again) {
          ax = ro.ax; ay = ro.ay; dir = ro.dir; carry = 0; steps = 0;
          if (PF) { tx = ro.tx; ty = ro.ty; flags = (flags & 0xFFu) | (ro.aux << 8); }
        }
        if (WIN && again) load_view_words(g, ax, ay, dir, vw, ldw);  // the regenerated level replaces the loaded words
      }
    }

    // LAYOUT_WINDOW: the view gather is one exposed HBM round trip per tile (18 % of the warps' time on FourRooms,
    // profiles/r02_final_kstep_fourrooms_summary.txt). The next tile's records and actions, requested at the top of
    // this tile, have arrived by now: ask L2 for the 7 lines that tile's gather will read (contiguous: 7 * lsw words),
    // so that the gather finds them a few hundred cycles away instead of in HBM. Hints only: a lane that regenerates
    // its env in the next tile prefetches lines it will not use.
    if (WIN && next < p.n_tiles) {
      const int axn = rec_n.x & 0xFF, ayn = (rec_n.x >> 8) & 0xFF, dn0 = rec_n.y & 3;
      const int dnn = stepping ? ((dn0 + (action_n == A_LEFT ? 3 : 0) + (action_n == A_RIGHT ? 1 : 0)) & 3) : dn0;
      const bool useCn = dnn & 1;
      const int lswn = useCn ? g.lswC : g.lswR;
      const uint32_t *w0 = p.grid + (size_t)(next * TILE + lane) * g.wpe + (useCn ? g.offC : 0) + ((useCn ? axn : ayn) - 3 + g.ring) * lswn;
      const int span = 7 * lswn * 4;  // bytes: 140 for FourRooms, at most 196
      asm volatile("prefetch.global.L2 [%0];" ::"l"(w0));
      asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char *>(w0) + span - 4));
      if (span > 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char *>(w0) + 128));
    }

    // ---- gen_obs ----
    if (obs != nullptr || packed_out != nullptr) {
      if (VIS == VIS_TBL && first) mbar_wait(tbl_bar, 0);  // the visibility table, requested in the prologue
      uint32_t clo[VIEW], chi[VIEW];
      if (WIN) {
        gather_from_words<VIS>(g, vw, vis_tbl, ax, ay, dir, carry, clo, chi);
      } else {
        const AccTiled acc = {base, true};
        gather_view<VIS>(g, acc, vis_tbl, ax, ay, dir, carry, clo, chi);
      }
      const int nvalid = min(TILE, p.n_envs - tile * TILE);
      if (packed_out == nullptr) {
        uint32_t S[OBS_WORDS];
        encode_stream(lut, clo, chi, S);
        // stage the 32 images in output layout in the consumed buffer, then ONE bulk store of the 4704-byte block.
        // (The ragged last tile / an unaligned obs pointer copy the valid bytes out of the stage instead: keeping the
        // stream words out of any byte-store path stops the compiler from spilling S to local memory on every tile.)
        const uint32_t n0 = __shfl_down_sync(0xFFFFFFFFu, S[0], 1);
        __syncwarp();  // orders memory among the lanes: every lane is past its tile / window reads before the stage overwrites them
        emit_obs_staged(gtile, lane, S, n0);
        if (nvalid == TILE && (obs_tma_ok & 1)) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            tma_store_1d(obs + (size_t)tile * OBS_TILE_BYTES, smem_u32(gtile), OBS_TILE_BYTES);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        } else {
          __syncwarp();
          const uint8_t *sbytes = reinterpret_cast<const uint8_t *>(gtile);
          uint8_t *dst = obs + (size_t)tile * OBS_TILE_BYTES;
          for (int i = lane; i < nvalid * OBS_BYTES; i += 32) dst[i] = sbytes[i];
        }
      } else {
        // host path, MG_HOST_PACKED: 13 words per env (cell codes + flags + step count) instead of the 147-byte image
        // and the four result arrays; the host expands them (mg_host_expand.cpp)
        uint32_t P[PACKED_WORDS];
        const uint32_t rewarded = reward != 0.0 ? 1u : 0u;
        if (rewarded && (uint32_t)rsteps >= PACKED_MAX_STEPS) atomicOr(p.err, ERR_PACKED_RANGE);
        // (the only negative reward, Dynamic-Obstacles' -1, travels as the reserved step count PACKED_MAX_STEPS)
        pack_codes(clo, chi, packed_tail(dir, terminated, truncated, rewarded, reward < 0.0 ? PACKED_MAX_STEPS : (uint32_t)rsteps), P);
        __syncwarp();
        uint32_t *dstw = gtile + PACKED_WORDS * lane;  // odd word stride: conflict-free
#pragma unroll
        for (int j = 0; j < PACKED_WORDS; ++j) dstw[j] = P[j];
        if (nvalid == TILE) {
          asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
          __syncwarp();
          if (lane == 0) {
            tma_store_1d(packed_out + (size_t)tile * (PACKED_WORDS * TILE), smem_u32(gtile), PACKED_TILE_BYTES);
            asm volatile("cp.async.bulk.commit_group;" ::: "memory");
          }
        } else {
          __syncwarp();
          uint32_t *dst = packed_out + (size_t)tile * (PACKED_WORDS * TILE);
          for (int i = lane; i < nvalid * PACKED_WORDS; i += 32) dst[i] = gtile[i];
        }
      }
    }
    if (active) {
      if (stepping) {
        rec.x = (uint32_t)ax | ((uint32_t)ay << 8);
        if (PF) rec.x |= ((uint32_t)tx << 16) | ((uint32_t)ty << 24);
        rec.y = (uint32_t)dir | (flags << 8);
        rec.z = carry;
        rec.w = (uint32_t)steps;
        p.agent[env] = rec;
      }
      if (dir_out) dir_out[env] = dir;
      if (reward_out) reward_out[env] = reward;
      if (term_out) term_out[env] = (uint8_t)terminated;
      if (trunc_out) trunc_out[env] = (uint8_t)truncated;
    }
    if (stepping && p.mode == AUTORESET_NEXT_STEP) {
      // scheduling hint (see ORDER_CAP). bit 0: an env of the tile ended in this step, so the tile regenerates in the
      // next one; bit 1: one will be truncated in the next step, so the tile regenerates in the step after. The next
      // launch reads these flags in its prologue, while this launch's last tiles are still being processed: a tile whose
      // byte is still the previous step's then shows its bit 1, which is exactly the truncation it missed.
      const unsigned anyp = __ballot_sync(0xFFFFFFFFu, active && (flags & FLAG_PENDING));
      const unsigned soon = __ballot_sync(0xFFFFFFFFu, active && !(flags & FLAG_PENDING) && steps + 1 >= p.max_steps);
      if (lane == 0) p.tile_hot[tile] = (uint8_t)((anyp ? 1 : 0) | (soon ? 2 : 0));
    }
    __syncwarp();  // lanes may still be reading this buffer (partial-tile path) before it is refilled
#ifdef MG_TIMELINE
    if (first) MG_TL(4);
    if (lane == 0) {
      unsigned long long *tl = g_tl[(obs_tma_ok >> 1) & 1][blockIdx.x];
      const unsigned long long t1 = gtime();
      if (tl_hot) { atomicAdd(&tl[8], 1ull); atomicMax(&tl[9], t1 - tl_t0); atomicMax(&tl[11], t1); atomicMax(&tl[12], (unsigned long long)(tile - t_lo)); }
      else atomicMax(&tl[10], t1 - tl_t0);
    }
#endif
    first = false;
    if (WIN) {
      if (stepping && next < p.n_tiles && ((rec_n.y >> 8) & FLAG_PENDING)) prefetch_rng(p.rng + (size_t)next * TILE + lane);
      tile = next;
      next = __shfl_sync(0xFFFFFFFFu, nn, 0);
      rec = rec_n;
      action = action_n;
    } else {
      if (lane == 0) nn = map_tile(atomicAdd(s_next, 1));
      tile = __shfl_sync(0xFFFFFFFFu, nn, 0);
    }
  }
  if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
  // the visibility table's bulk copy must have landed before the CTA's shared memory is released (a CTA without
  // tiles, or an observation-less pass, never waited for it)
  if (VIS == VIS_TBL && threadIdx.x == 0) mbar_wait(tbl_bar, 0);
  MG_TL(5);
  MG_TL_EXIT();
}


typedef void (*StepKernel)(Params, const void *, int, uint8_t *, int32_t *, double *, uint8_t *, uint8_t *, uint32_t *, int);

template <int VIS, int LAYOUT>
static StepKernel pick_kind(int kind) {
  switch (kind) {
    case KIND_EMPTY: return (StepKernel)k_step<KIND_EMPTY, VIS, LAYOUT>;
    case KIND_DOORKEY: return (StepKernel)k_step<KIND_DOORKEY, VIS, LAYOUT>;
    case KIND_CROSSING: return (StepKernel)k_step<KIND_CROSSING, VIS, LAYOUT>;
    case KIND_LAVAGAP: return (StepKernel)k_step<KIND_LAVAGAP, VIS, LAYOUT>;
    case KIND_DISTSHIFT: return (StepKernel)k_step<KIND_DISTSHIFT, VIS, LAYOUT>;
    case KIND_MULTIROOM: return (StepKernel)k_step<KIND_MULTIROOM, VIS, LAYOUT>;
    case KIND_LOCKEDROOM: return (StepKernel)k_step<KIND_LOCKEDROOM, VIS, LAYOUT>;
    case KIND_PLAYGROUND: return (StepKernel)k_step<KIND_PLAYGROUND, VIS, LAYOUT>;
    case KIND_GOTODOOR: return (StepKernel)k_step<KIND_GOTODOOR, VIS, LAYOUT>;
    case KIND_FETCH: return (StepKernel)k_step<KIND_FETCH, VIS, LAYOUT>;
    case KIND_REDBLUEDOORS: return (StepKernel)k_step<KIND_REDBLUEDOORS, VIS, LAYOUT>;
    case KIND_GOTOOBJECT: return (StepKernel)k_step<KIND_GOTOOBJECT, VIS, LAYOUT>;
    case KIND_PUTNEAR: return (StepKernel)k_step<KIND_PUTNEAR, VIS, LAYOUT>;
    case KIND_MEMORY: return (StepKernel)k_step<KIND_MEMORY, VIS, LAYOUT>;
    case KIND_DYNOBS: return (StepKernel)k_step<KIND_DYNOBS, VIS, LAYOUT>;
    case KIND_ROOMGRID: return (StepKernel)k_step<KIND_ROOMGRID, VIS, LAYOUT>;
    default: return (StepKernel)k_step<KIND_FOURROOMS, VIS, LAYOUT>;
  }
}
template <int LAYOUT>
static StepKernel pick_vis(int kind, int vis) {
  return vis == VIS_NONE ? pick_kind<VIS_NONE, LAYOUT>(kind) : pick_kind<VIS_TBL, LAYOUT>(kind);
}

StepKernel step_kernel_window(int kind, int vis);  // mg_step_window.cu

}  // namespace mg
