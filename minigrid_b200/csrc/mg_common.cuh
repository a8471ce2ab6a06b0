// mg_common.cuh — device data layout shared by every kernel of the engine.
//
// The reference's per-env object graph (Grid = list[WorldObj|None], minigrid/core/grid.py:35; WorldObj with
// type/color/is_open/is_locked, core/world_object.py:27-43,171-176) becomes:
//
//   cell code (1 byte)   bits 0-3  t4     = OBJECT_TO_IDX type (core/constants.py:25-37) with the door state
//                                           folded in: 4 door open, 11 door closed, 12 door locked
//                        bits 4-6  colour = COLOR_TO_IDX (core/constants.py:20)
//                        bit  7    opaque = !see_behind() (world_object.py:57,164,181), kept redundantly so
//                                           that Grid.process_vis's transparency test is one bit
//   grid tile            32 consecutive envs ("one warp-lane per environment"), word-interleaved:
//                        tile[w][lane] uint32, w < wpe. Lane L's w-th word sits in shared-memory bank L, so
//                        per-lane gathers at lane-specific offsets are conflict-free, and a tile is one
//                        contiguous block that a single TMA bulk copy (cp.async.bulk) stages.
//   per env words        array R: lines y = -ring..H+ring-1 (row-major x bytes, ring lines are grey wall), then
//                        array C: lines x = -ring..W+ring-1 (column-major y bytes): every 7-cell run of the
//                        egocentric view (Grid.slice + rotate_left, grid.py:110-143) is 7 consecutive
//                        bytes of one line of R (facing +-x) or C (facing +-y).
//   agent record         uint4 {x | y<<8, dir | flags<<8, carry code (0 none), step_count}
//   rng record           numpy PCG64 bit-generator state (state, inc, has_uint32, uinteger)
#pragma once
#include <stdint.h>
#ifdef __CUDACC__
#include <cuda_runtime.h>
#define MG_HD __host__ __device__ __forceinline__
#define MG_D __device__ __forceinline__
#else
// Host build of the per-lane logic (tests/host_emu only: a CPU check of the device arithmetic before GPU time
// is spent; never part of the product library). The shim supplies uint4 and the few intrinsics used below.
#include "mg_host_shim.h"
#define MG_HD inline
#define MG_D inline
#endif

namespace mg {

constexpr int VIEW = 7;
constexpr int OBS_BYTES = 147;
constexpr int TILE = 32;                    // envs per tile == lanes per warp
constexpr int OBS_TILE_BYTES = OBS_BYTES * TILE;  // 4704, a multiple of 16
constexpr int OBS_WORDS = 37;               // ceil(147 / 4)
constexpr int MAX_DIM = 26;                 // W, H <= 26 (the OOB bit mask is built in 32 bits)

// core/constants.py:25-37
enum : uint32_t { T_UNSEEN = 0, T_EMPTY = 1, T_WALL = 2, T_FLOOR = 3, T_DOOR = 4, T_KEY = 5, T_BALL = 6,
                  T_BOX = 7, T_GOAL = 8, T_LAVA = 9, T_AGENT = 10, T4_DOOR_CLOSED = 11, T4_DOOR_LOCKED = 12,
                  // Box.contains (world_object.py:273-293) is None everywhere except ObstructedMaze, whose grey boxes hide
                  // the key of a door: t4 = 13 is "a grey box with a key inside", the colour field is the KEY's colour
                  T4_BOX_WITH_KEY = 13 };
enum : uint32_t { C_RED = 0, C_GREEN = 1, C_BLUE = 2, C_PURPLE = 3, C_YELLOW = 4, C_GREY = 5 };
// core/actions.py:7-20
enum : int { A_LEFT = 0, A_RIGHT = 1, A_FORWARD = 2, A_PICKUP = 3, A_DROP = 4, A_TOGGLE = 5, A_DONE = 6 };

constexpr uint32_t OPAQUE_BIT = 0x80u;
constexpr uint32_t CODE_EMPTY = T_EMPTY;
constexpr uint32_t CODE_WALL = T_WALL | (C_GREY << 4) | OPAQUE_BIT;  // 0xD2, Wall() (world_object.py:160-162)
constexpr uint32_t CODE_WALL4 = CODE_WALL * 0x01010101u;
constexpr uint32_t CODE_GOAL = T_GOAL | (C_GREEN << 4);
constexpr uint32_t CODE_LAVA = T_LAVA | (C_RED << 4);

// agent flags (second word of the agent record, bits 8..)
constexpr uint32_t FLAG_PENDING = 2u;  // episode ended last step (SyncVectorEnv._autoreset_envs[i], NEXT_STEP)

enum : int { KIND_EMPTY = 0, KIND_DOORKEY = 1, KIND_CROSSING = 2, KIND_FOURROOMS = 3, KIND_LAVAGAP = 4, KIND_DISTSHIFT = 5,
             KIND_MULTIROOM = 6,
             // SURVEY 8(f-1) and 8(f-2), next: the generators (mg_levels.cuh) and step post-filters (mg_postfilter.cuh) of
             // the kinds below exist and are checked against the oracle on the CPU (tests/test_oracle_next.py); K1 / K2
             // are not instantiated for them yet and mg_create rejects them (KIND_COUNT)
             KIND_LOCKEDROOM = 7, KIND_PLAYGROUND = 8,
             KIND_GOTODOOR = 9, KIND_FETCH = 10, KIND_REDBLUEDOORS = 11, KIND_GOTOOBJECT = 12, KIND_PUTNEAR = 13,
             KIND_MEMORY = 14,
             // SURVEY 8(f-4): RNG draws inside step (envs/dynamicobstacles.py)
             KIND_DYNOBS = 15,
             // SURVEY 8(f-2), second half: core/roomgrid.py with unlock.py, unlockpickup.py, blockedunlockpickup.py, keycorridor.py
             KIND_ROOMGRID = 16 };
constexpr int KIND_COUNT = 17;
// kp[0] of KIND_ROOMGRID; the ObstructedMaze variants (envs/obstructedmaze.py, obstructedmaze_v1.py) also read
// kp[4] key_in_box, kp[5] blocked, kp[6] agent room i | j << 4, kp[7] num_quarters
enum : int { RG_UNLOCK = 0, RG_UNLOCKPICKUP = 1, RG_BLOCKEDUNLOCKPICKUP = 2, RG_KEYCORRIDOR = 3, RG_OBSTRUCTED_1D = 4,
             RG_OBSTRUCTED_FULL = 5, RG_OBSTRUCTED_FULL_V1 = 6 };  // kinds mg_create accepts: the kernels are instantiated for the kinds below this
enum : int { AUTORESET_NEXT_STEP = 0, AUTORESET_SAME_STEP = 1, AUTORESET_DISABLED = 2 };
// bits of the sticky device error word (Params::err)
enum : int { ERR_BAD_ACTION = 1, ERR_BAD_STATE = 2, ERR_PACKED_RANGE = 4 };

// (type, colour, state) -> cell code. None/unseen/agent all mean "no object" (WorldObj.decode,
// world_object.py:77-78) and encode as (1,0,0) (grid.py:258-261).
MG_HD uint32_t encode_cell(uint32_t type, uint32_t color, uint32_t state) {
  if (type == T_EMPTY || type == T_UNSEEN || type >= T_AGENT) return CODE_EMPTY;
  uint32_t t4 = type, opaque = 0;
  if (type == T_DOOR) {
    t4 = state == 0 ? (uint32_t)T_DOOR : (state == 1 ? (uint32_t)T4_DOOR_CLOSED : (uint32_t)T4_DOOR_LOCKED);
    opaque = state != 0;
  } else if (type == T_WALL) {
    opaque = 1;
  }
  return t4 | ((color & 7u) << 4) | (opaque << 7);
}
// cell code -> type | colour << 8 | state << 16 (WorldObj.encode / Door.encode, world_object.py:65-67,196-212)
MG_HD uint32_t decode_cell(uint32_t code) {
  uint32_t t4 = code & 15u, color = (code >> 4) & 7u;
  if (t4 == T_UNSEEN) return 0;
  if (t4 == T_EMPTY) return T_EMPTY;
  if (t4 == T4_DOOR_CLOSED) return T_DOOR | (color << 8) | (1u << 16);
  if (t4 == T4_DOOR_LOCKED) return T_DOOR | (color << 8) | (2u << 16);
  if (t4 == T4_BOX_WITH_KEY) return T_BOX | (C_GREY << 8);  // what is inside does not show (Box.encode is WorldObj.encode)
  return t4 | (color << 8);
}

// Two HBM layouts of the per-env words (same words, same r_word / c_word indices):
//   LAYOUT_TILED   tile[w][lane] for 32 consecutive envs (small grids): one TMA bulk copy stages a whole tile and
//                  per-lane gathers are bank-conflict free.
//   LAYOUT_WINDOW  env-major, lines of ceil(W / 4) words, 3 ring lines (large grids): a step only touches the 7 lines of
//                  the egocentric view, contiguous in one array, which each lane gathers straight into registers;
//                  HBM traffic per env-step grows with the grid's side, not its area.
enum : int { LAYOUT_TILED = 0, LAYOUT_WINDOW = 1 };
constexpr int WIN_LANE_BYTES = 240; // (host emulation of the round-1 window staging only)

struct Geom {
  int W, H;
  int lswR, lswC;  // words per line of R / C
  int ring;        // wall lines stored before line 0 and after the last line of each array
  int offC;        // word offset of array C inside an env
  int wpe;         // words per env
  int layout;
};

MG_HD Geom make_geom(int W, int H, int layout) {
  Geom g;
  g.W = W; g.H = H; g.layout = layout;
  if (layout == LAYOUT_TILED) { g.lswR = (W + 3) >> 2; g.lswC = (H + 3) >> 2; g.ring = 1; }
  else { g.lswR = (W + 3) >> 2; g.lswC = (H + 3) >> 2; g.ring = 3; }  // lines as wide as the grid: a step's 7 lines are 7 * lsw words
  g.offC = (H + 2 * g.ring) * g.lswR;
  g.wpe = g.offC + (W + 2 * g.ring) * g.lswC;
  if (layout != LAYOUT_TILED) {  // both arrays of every env start on 16 bytes (K3 stages array C with bulk copies)
    g.offC = (g.offC + 3) & ~3;
    g.wpe = (g.offC + (W + 2 * g.ring) * g.lswC + 3) & ~3;
  }
  return g;
}
// index in the grid arena (in words) of word w of environment env
MG_HD size_t grid_word(const Geom &g, int env, int w) {
  return g.layout == LAYOUT_TILED ? ((size_t)(env >> 5) * g.wpe + w) * 32 + (env & 31) : (size_t)env * g.wpe + w;
}

struct RngRec {  // 48 bytes, 16-byte aligned
  uint64_t state_hi, state_lo, inc_hi, inc_lo;
  uint32_t has_uint32, uinteger;
  uint64_t pad;
};

struct Params {
  Geom g;
  int n_envs, n_tiles;
  int max_steps, see_through, mode, kind;
  int kp[8];                // generator parameters (see include/minigrid_b200.h)
  uint32_t *grid;           // n_tiles * 32 * wpe words, see grid_word()
  uint4 *agent;             // [n_tiles * 32]
  uint4 *extra;             // [n_tiles * 32], KIND_DYNOBS only: the obstacles in list order, 16 bits each (x | y << 8)
  RngRec *rng;              // [n_tiles * 32]
  const double *reward_lut; // [max_steps + 1], 1 - 0.9 * (k / max_steps) computed on the host in IEEE double
  const uint32_t *cell_lut; // [256] decode_cell()
  const uint16_t *vis_tbl;  // [128 * 128] process_vis row table (mg_obs.cuh: build_vis_table)
  const uint32_t *tmpl;     // [wpe] level template: the words of a blank draw (mg_levels.cuh)
  int *err;                 // sticky error word
  uint8_t *tile_hot;        // [n_tiles] 1 = an env of the tile ended in the last step (K1's scheduling hint, never semantics)
  // the reference's reward wrappers around every env (wrappers.py:68-184, 809-882), 0 = absent
  int no_death_mask;        // NoDeath: bit t = OBJECT_TO_IDX type t is a death cell
  int bonus_mode;           // 1 ActionBonus, 2 PositionBonus
  double death_cost;        // NoDeath.death_cost
  uint32_t *counts;         // [n_envs][W * H * 28] (ActionBonus) or [n_envs][W * H] (PositionBonus): the wrappers' self.counts
};

struct StepPlan {  // launch shape of K1, chosen once per handle (mg_step.cu: configure_step)
  int warps, vis, ctas_per_sm, grid;
  size_t smem;
};

// word index of byte (line, pos) and helpers for the interleaved tile
MG_HD int r_word(const Geom &g, int x, int y) { return (y + g.ring) * g.lswR + (x >> 2); }
MG_HD int c_word(const Geom &g, int x, int y) { return g.offC + (x + g.ring) * g.lswC + (y >> 2); }
// byte offsets in the grid arena of cell (x, y) in the two arrays
MG_HD size_t cell_byte_R(const Geom &g, int env, int x, int y) { return grid_word(g, env, r_word(g, x, y)) * 4 + (x & 3); }
MG_HD size_t cell_byte_C(const Geom &g, int env, int x, int y) { return grid_word(g, env, c_word(g, x, y)) * 4 + (y & 3); }

// PTX prmt.b32 (generic mode): selector nibble bits 0-2 pick one of the 8 source bytes, bit 3 replicates that
// byte's sign bit instead. CUDA's __byte_perm() only honours the low 3 bits, hence the inline PTX.
MG_D uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
#ifdef __CUDA_ARCH__
  uint32_t d;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
  return d;
#else
  return __byte_perm(a, b, sel);
#endif
}
MG_HD int clampi(int v, int lo, int hi) { return v < lo ? lo : (v > hi ? hi : v); }
// bit i (i < 4) -> bit 8i
MG_HD uint32_t spread4(uint32_t b) { return (b * 0x00204081u) & 0x01010101u; }

#ifdef __CUDACC__
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
#endif

}  // namespace mg
