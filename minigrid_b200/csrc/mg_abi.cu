// mg_abi.cu — the C-ABI of include/minigrid_b200.h: handle management, launch sequencing (autoreset
// modes), and the host-buffer (end-to-end) entry points. No torch types cross this boundary.
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/minigrid_b200.h"
#include "mg_common.cuh"
#include "mg_obs.cuh"
#include "mg_host_expand.h"

namespace mg {
cudaError_t launch_step(const Params &p, const StepPlan &plan, const void *actions, int action_dtype, uint8_t *obs,
                        int32_t *dir, double *reward, uint8_t *term, uint8_t *trunc, uint32_t *packed, int step_parity,
                        cudaStream_t stream);
cudaError_t configure_step(const Params &p, StepPlan *plan);
cudaError_t launch_reset(const Params &p, const uint8_t *mask, uint8_t *obs, int32_t *dir, cudaStream_t stream);
cudaError_t launch_seed(const Params &p, const uint8_t *mask, const uint64_t *seeds_dev, uint64_t base, cudaStream_t stream);
cudaError_t launch_full_obs(const Params &p, uint8_t *out, int with_agent, cudaStream_t stream);
cudaError_t launch_get_state(const Params &p, uint8_t *grid, int32_t *agent, uint64_t *rng, uint8_t *pending,
                             cudaStream_t stream);
cudaError_t launch_set_state(const Params &p, const uint8_t *grid, const int32_t *agent, const uint64_t *rng,
                             const uint8_t *pending, cudaStream_t stream);
cudaError_t launch_init(const Params &p, cudaStream_t stream);
cudaError_t launch_clear_err(const Params &p, int bits, cudaStream_t stream);
cudaError_t launch_view(const Params &p, int V, uint8_t *out, cudaStream_t s);
cudaError_t launch_onehot(const uint8_t *img, uint8_t *out, long long n_cells, cudaStream_t s);
cudaError_t launch_flat(const uint8_t *img, const uint8_t *mission, uint8_t *out, int img_bytes, int mission_bytes, long long n_envs,
                        cudaStream_t s);
cudaError_t launch_symbolic(const Params &p, long long *out, cudaStream_t s);
cudaError_t launch_rgb_partial(const uint8_t *img, const uint8_t *tiles, const uint16_t *index, uint8_t *out, long long n_envs, cudaStream_t s);
cudaError_t launch_rgb_full(const Params &p, const uint8_t *img, const uint8_t *tiles, const uint16_t *index, uint8_t *out, cudaStream_t s);
cudaError_t launch_template(const Params &p, uint32_t *tmpl, cudaStream_t stream);
}  // namespace mg

using namespace mg;

struct mg_env {
  Params p;
  int device;
  StepPlan plan;     // launch shape of K1
  int64_t launches;
  // device allocations owned by the handle
  void *d_arena;     // grid | agent | rng | lists | counts | err | luts, one cudaMalloc
  uint64_t *d_seeds;
  // host path
  cudaStream_t hstream;
  cudaStream_t last_stream; int has_last_stream;  // last caller stream that touched the handle's state
  cudaEvent_t ev_order;                            // orders hstream (the *_host entry points) after that stream
  int32_t *d_actions; uint8_t *d_out;  // device mirror of the host-facing buffers
  int32_t *h_actions; uint8_t *h_out;  // pinned staging, used when the caller's buffers are pageable
  int *h_err;
  // MG_HOST_PACKED: 52-byte step records cross PCIe in chunks and are expanded by a pool of host threads
  int host_format;
  uint32_t *d_packed; uint8_t *h_packed;   // device records, pinned landing buffer
  double *h_reward_lut;                    // host copy of the reward table
  int pool_threads;                        // what this handle asked for (the pool itself is process-wide)
  cudaEvent_t chunk_ev[16];
  int n_chunks;
  // store form of the host expansion (mg_host_expand.cpp: expand_range): calibrated per handle, because it depends on
  // whether the caller's output arrays stay in the host's last-level cache. A calibration is ten steps with plain stores,
  // then ten with streaming stores (blocks, not alternation: plain stores only win once the arrays ARE cache-resident,
  // which a streaming step in between undoes); the last six calls of each block are timed and the faster form is kept
  // for the next 8192 steps.
  int stream_fixed;            // -1 calibrate, 0 / 1 forced by MINIGRID_B200_EXPAND_STREAM
  int stream_mode;             // the form in use outside a calibration
  int64_t packed_steps;        // packed host steps so far
  double cal_us[2]; int cal_n[2];
  // MINIGRID_B200_HOST_TRACE=1: where a packed host step spends its time (printed by mg_destroy)
  int trace; double tr_enqueue, tr_first_chunk, tr_last_chunk, tr_pool, tr_total; int64_t tr_n;
  // optional per-launch timing of K1 (bench.py's roofline leg)
  int profiling;
  std::vector<cudaEvent_t> *prof_events;  // start/stop pairs
};

static thread_local std::string g_err;

// The host threads that expand packed step records are ONE pool per process, shared by every handle: a training process
// that cycles through several handles (bench.py rotates four) must not keep four sets of workers spinning. A step takes
// the pool for its duration; handles driven from different host threads serialise on it.
static std::mutex g_pool_mu;       // guards g_pool and serialises its use
static HostPool *g_pool = nullptr;
const char *mg_last_error(void) { return g_err.c_str(); }

static int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define MG_CUDA(call)                                                                          \
  do {                                                                                         \
    cudaError_t e__ = (call);                                                                  \
    if (e__ != cudaSuccess)                                                                    \
      return fail(MG_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));          \
  } while (0)

static size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// Every entry point works on the handle's device and leaves the calling thread's current device as it found it
// (a process that steps an env on cuda:1 and runs its policy on cuda:0 must not see its current device change,
// also not when a handle is destroyed from a garbage collector).
struct DeviceGuard {
  int prev = -1, dev;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) : dev(device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != dev) err = cudaSetDevice(dev);
  }
  ~DeviceGuard() {
    if (prev >= 0 && prev != dev) cudaSetDevice(prev);
  }
};
#define MG_ON_DEVICE(h)            \
  DeviceGuard guard__((h)->device); \
  MG_CUDA(guard__.err)

int mg_create(int kind, int width, int height, int max_steps, int see_through_walls, const int32_t *params,
              int n_params, int64_t n_envs, int autoreset_mode, int device, mg_env **out) {
  if (!out) return fail(MG_ERR_INVALID_ARG, "out is NULL");
  *out = nullptr;
  if (kind < 0 || kind >= KIND_COUNT) return fail(MG_ERR_INVALID_ARG, "unknown kind");
  if (width < 3 || height < 3 || width > MAX_DIM || height > MAX_DIM)
    return fail(MG_ERR_INVALID_ARG, "width/height must be in [3, 26]");
  if (max_steps < 1) return fail(MG_ERR_INVALID_ARG, "max_steps must be >= 1");
  if (n_envs < 1 || n_envs > (int64_t)1 << 30) return fail(MG_ERR_INVALID_ARG, "n_envs out of range");
  if (autoreset_mode < 0 || autoreset_mode > 2) return fail(MG_ERR_INVALID_ARG, "unknown autoreset mode");
  if ((kind == MG_KIND_FETCH || kind == MG_KIND_GOTOOBJECT || kind == MG_KIND_PUTNEAR) &&
      (n_params < 1 || params[0] < 1 || params[0] > 8))
    return fail(MG_ERR_INVALID_ARG, "fetch / gotoobject / putnear need params {numObjs}, 1 <= numObjs <= 8");
  if (kind == MG_KIND_GOTODOOR && (width < 5 || height < 5))
    return fail(MG_ERR_INVALID_ARG, "gotodoor needs at least 5 x 5 (gotodoor.py:66)");
  if (kind == MG_KIND_REDBLUEDOORS && (width != 2 * height || height < 4))
    return fail(MG_ERR_INVALID_ARG, "redbluedoors is 2 size x size (redbluedoors.py:60-72)");
  if (kind == MG_KIND_MEMORY && (height % 2 == 0 || height < 7 || width < 7))
    return fail(MG_ERR_INVALID_ARG, "memory needs an odd height and at least 7 x 7 (memory.py:98)");
  if (kind == MG_KIND_ROOMGRID) {
    if (n_params < 4 || params[0] < 0 || params[0] > 6 || params[1] < 3 || params[1] > 8 || params[2] < 1 || params[3] < 1 ||
        params[2] * params[3] > 9 || width != (params[1] - 1) * params[3] + 1 || height != (params[1] - 1) * params[2] + 1)
      return fail(MG_ERR_INVALID_ARG, "roomgrid needs params {variant 0..3, room_size 3..8, num_rows, num_cols} with at most 9 rooms, "
                                      "width = (room_size - 1) num_cols + 1 and height = (room_size - 1) num_rows + 1 (roomgrid.py:83-84)");
    if (params[0] == 3 && params[3] != 3) return fail(MG_ERR_INVALID_ARG, "keycorridor has 3 columns of rooms (keycorridor.py:104-126)");
    if (params[0] != 3 && params[0] < 5 && (params[2] != 1 || params[3] != 2))
      return fail(MG_ERR_INVALID_ARG, "unlock / unlockpickup / blockedunlockpickup / obstructedmaze-1D are 1 x 2 rooms");
    if (params[0] >= 4) {
      if (n_params < 8 || params[1] < 4) return fail(MG_ERR_INVALID_ARG, "obstructedmaze needs params {variant, room_size >= 4, num_rows, num_cols, key_in_box, blocked, agent_room_i | agent_room_j << 4, num_quarters}");
      if (params[0] >= 5 && (params[2] != 3 || params[3] != 3 || params[7] < 1 || params[7] > 4 || (params[6] & 15) > 2 || (params[6] >> 4) > 2))
        return fail(MG_ERR_INVALID_ARG, "obstructedmaze-Full is 3 x 3 rooms with 1..4 quarters and the agent's room inside the grid");
    }
    if (params[0] == 2 && params[1] < 4) return fail(MG_ERR_INVALID_ARG, "blockedunlockpickup needs room_size >= 4 (a cell in front of the door)");
  }
  if (kind == MG_KIND_DYNOBS) {
    if (n_params < 5 || params[0] < 0 || params[0] > 8)
      return fail(MG_ERR_INVALID_ARG, "dynamic obstacles need params {n_obstacles (0..8), random_start, start_x, start_y, start_dir}");
    if (width > 16 || height > 16) return fail(MG_ERR_INVALID_ARG, "dynamic obstacles: at most 16 x 16 (the obstacles move inside the staged tile)");
  }
  if (kind == MG_KIND_LOCKEDROOM && (width != height || width < 13))
    return fail(MG_ERR_INVALID_ARG, "lockedroom needs a square grid of at least 13 x 13 (lockedroom.py:108-173)");
  if (kind == MG_KIND_PLAYGROUND && (width != 19 || height != 19))
    return fail(MG_ERR_INVALID_ARG, "playground is 19 x 19 (playground.py:16-25)");
  if (kind == MG_KIND_CROSSING && (width % 2 == 0 || height % 2 == 0))
    return fail(MG_ERR_INVALID_ARG, "crossing needs odd sizes (crossing.py:132)");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(MG_ERR_NO_DEVICE, "no CUDA device: the engine has no CPU fallback");
  if (device < 0) MG_CUDA(cudaGetDevice(&device));
  if (device >= ndev) return fail(MG_ERR_INVALID_ARG, "device index out of range");
  DeviceGuard guard(device);
  MG_CUDA(guard.err);

  mg_env *h = new (std::nothrow) mg_env();
  if (!h) return fail(MG_ERR_INVALID_ARG, "out of host memory");
  memset(h, 0, sizeof(*h));
  Params &p = h->p;
  {
    // small grids: whole tiles through TMA; large grids: env-major lines and per-lane view windows (mg_common.cuh)
    int layout = make_geom(width, height, LAYOUT_TILED).wpe * 4 > 512 ? LAYOUT_WINDOW : LAYOUT_TILED;
    if (const char *e = getenv("MINIGRID_B200_LAYOUT")) layout = atoi(e) ? LAYOUT_WINDOW : LAYOUT_TILED;  // tuning / test knob
    if (kind == MG_KIND_DYNOBS) layout = LAYOUT_TILED;  // its obstacles move through cells all over the grid: whole tiles only
    p.g = make_geom(width, height, layout);
  }
  p.n_envs = (int)n_envs;
  p.n_tiles = (int)((n_envs + TILE - 1) / TILE);
  p.max_steps = max_steps;
  p.see_through = see_through_walls ? 1 : 0;
  p.mode = autoreset_mode;
  p.kind = kind;
  h->trace = getenv("MINIGRID_B200_HOST_TRACE") != nullptr;
  h->stream_fixed = -1;
  if (const char *es = getenv("MINIGRID_B200_EXPAND_STREAM")) h->stream_fixed = atoi(es) != 0;
  for (int i = 0; i < 8; ++i) p.kp[i] = (params && i < n_params) ? params[i] : 0;
  if (kind == MG_KIND_EMPTY && !p.kp[0] && n_params < 4) { p.kp[1] = 1; p.kp[2] = 1; p.kp[3] = 0; }
  if (kind == MG_KIND_CROSSING && n_params < 2) { p.kp[0] = 1; p.kp[1] = (int)T_LAVA; }
  if (kind == MG_KIND_LAVAGAP && n_params < 1) p.kp[0] = (int)T_LAVA;
  if (kind == MG_KIND_MULTIROOM) {
    if (n_params < 3) p.kp[2] = 10;
    if (p.kp[0] < 1 || p.kp[1] < p.kp[0] || p.kp[1] > 6 || p.kp[2] < 4 || p.kp[2] > 10) {
      delete h;
      return fail(MG_ERR_INVALID_ARG, "multiroom: need 1 <= minNumRooms <= maxNumRooms <= 6 and 4 <= maxRoomSize <= 10");
    }
  }
  if (kind == MG_KIND_DISTSHIFT && n_params < 4) { if (n_params < 1) p.kp[0] = 2; p.kp[1] = 1; p.kp[2] = 1; p.kp[3] = 0; }
  // a fixed agent start (agent_start_pos / agent_start_dir, empty.py:75-76, distshift.py:68-69) must lie inside the
  // border walls: K1 trusts the agent record
  if (kind == MG_KIND_DYNOBS && !p.kp[1] &&
      (p.kp[2] < 1 || p.kp[2] > width - 2 || p.kp[3] < 1 || p.kp[3] > height - 2 || p.kp[4] < 0 || p.kp[4] > 3)) {
    delete h;
    return fail(MG_ERR_INVALID_ARG, "agent start must satisfy 1 <= x <= width - 2, 1 <= y <= height - 2, 0 <= dir <= 3");
  }
  if ((kind == MG_KIND_EMPTY && !p.kp[0]) || kind == MG_KIND_DISTSHIFT) {
    if (p.kp[1] < 1 || p.kp[1] > width - 2 || p.kp[2] < 1 || p.kp[2] > height - 2 || p.kp[3] < 0 || p.kp[3] > 3) {
      delete h;
      return fail(MG_ERR_INVALID_ARG, "agent start must satisfy 1 <= x <= width - 2, 1 <= y <= height - 2, 0 <= dir <= 3");
    }
  }
  h->device = device;

  const size_t n_pad = (size_t)p.n_tiles * TILE;
  const size_t sz_grid = align_up((size_t)p.n_tiles * p.g.wpe * 128, 256) + 256;  // + slack: window copies read 224 B from a line start
  const size_t sz_agent = align_up(n_pad * sizeof(uint4), 256);
  const size_t sz_rng = align_up(n_pad * sizeof(RngRec), 256);
  const size_t sz_lut_r = align_up((size_t)(max_steps + 1) * sizeof(double), 256);
  const size_t sz_tmpl = align_up((size_t)p.g.wpe * 4, 256);
  const size_t sz_hot = align_up((size_t)p.n_tiles, 256);
  const size_t sz_extra = kind == MG_KIND_DYNOBS ? align_up(n_pad * sizeof(uint4), 256) : 0;
  const size_t total = sz_grid + sz_agent + sz_rng + 256 /*err*/ + sz_lut_r + 1024 + VIS_TBL_BYTES + sz_tmpl + sz_hot + sz_extra;
  cudaError_t e = cudaMalloc(&h->d_arena, total);
  if (e != cudaSuccess) { delete h; return fail(MG_ERR_CUDA, std::string("cudaMalloc arena: ") + cudaGetErrorString(e)); }
  uint8_t *base = (uint8_t *)h->d_arena;
  p.grid = (uint32_t *)base; base += sz_grid;
  p.agent = (uint4 *)base; base += sz_agent;
  p.rng = (RngRec *)base; base += sz_rng;
  p.err = (int *)base; base += 256;
  double *d_rl = (double *)base; base += sz_lut_r;
  uint32_t *d_cl = (uint32_t *)base; base += 1024;
  uint16_t *d_vt = (uint16_t *)base; base += VIS_TBL_BYTES;
  uint32_t *d_tm = (uint32_t *)base; base += sz_tmpl;
  p.tile_hot = base; base += sz_hot;
  p.extra = sz_extra ? (uint4 *)base : nullptr;
  p.reward_lut = d_rl; p.cell_lut = d_cl; p.vis_tbl = d_vt; p.tmpl = d_tm;

  // _reward(): 1 - 0.9 * (step_count / max_steps) in host IEEE double, never contracted (minigrid_env.py:245)
  {
    double *lut = (double *)malloc((size_t)(max_steps + 1) * sizeof(double));
    for (int k = 0; k <= max_steps; ++k) {
      volatile double q = (double)k / (double)max_steps;
      volatile double m = 0.9 * q;
      lut[k] = 1.0 - m;
    }
    e = cudaMemcpy(d_rl, lut, (size_t)(max_steps + 1) * sizeof(double), cudaMemcpyHostToDevice);
    h->h_reward_lut = lut;  // also the table of the host-side expansion (MG_HOST_PACKED)
    uint32_t cl[256];
    for (uint32_t c = 0; c < 256; ++c) cl[c] = decode_cell(c);
    if (e == cudaSuccess) e = cudaMemcpy(d_cl, cl, sizeof(cl), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemset(p.err, 0, 256);
    if (e == cudaSuccess) e = cudaMemset(p.tile_hot, 0, sz_hot);
    if (e == cudaSuccess && sz_extra) e = cudaMemset(p.extra, 0, sz_extra);
    uint16_t *vt = (uint16_t *)malloc(VIS_TBL_BYTES);
    build_vis_table(vt);
    if (e == cudaSuccess) e = cudaMemcpy(d_vt, vt, VIS_TBL_BYTES, cudaMemcpyHostToDevice);
    free(vt);
  }
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->hstream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaEventCreateWithFlags(&h->ev_order, cudaEventDisableTiming);
  if (e == cudaSuccess) e = configure_step(p, &h->plan);
  if (e == cudaSuccess && getenv("MINIGRID_B200_VERBOSE"))
    fprintf(stderr, "[minigrid_b200] K1 plan: layout=%d, %d warps/CTA, vis=%d, %d CTA/SM, grid=%d, smem=%zu B, tiles=%d\n", p.g.layout, h->plan.warps,
            h->plan.vis, h->plan.ctas_per_sm, h->plan.grid, h->plan.smem, p.n_tiles);
  if (e == cudaSuccess) e = launch_init(p, h->hstream);
  if (e == cudaSuccess) e = launch_template(p, d_tm, h->hstream);
  if (e == cudaSuccess) e = launch_seed(p, nullptr, nullptr, 0, h->hstream);
  if (e == cudaSuccess) e = cudaStreamSynchronize(h->hstream);
  if (e != cudaSuccess) {
    std::string msg = std::string("mg_create: ") + cudaGetErrorString(e);
    mg_destroy(h);
    return fail(MG_ERR_CUDA, msg);
  }
  h->launches = 3;
  *out = h;
  return MG_OK;
}

int mg_destroy(mg_env *h) {
  if (!h) return MG_OK;
  if (h->trace && h->tr_n)
    fprintf(stderr, "[minigrid_b200] packed host step, mean of %lld (us since entry): enqueued %.1f, first chunk on the host %.1f, last chunk %.1f, "
                    "expansion done %.1f, return %.1f; %d chunks, %d threads\n", (long long)h->tr_n, h->tr_enqueue / h->tr_n,
            h->tr_first_chunk / h->tr_n, h->tr_last_chunk / h->tr_n, h->tr_pool / h->tr_n, h->tr_total / h->tr_n, h->n_chunks,
            h->pool_threads);
  DeviceGuard guard(h->device);
  if (h->hstream) { cudaStreamSynchronize(h->hstream); cudaStreamDestroy(h->hstream); }
  if (h->ev_order) cudaEventDestroy(h->ev_order);
  cudaFree(h->d_arena);
  cudaFree(h->d_seeds);
  cudaFree(h->d_actions);
  cudaFree(h->d_out);
  cudaFreeHost(h->h_actions);
  cudaFreeHost(h->h_out);
  cudaFreeHost(h->h_err);
  cudaFree(h->d_packed);
  cudaFreeHost(h->h_packed);
  cudaFree(h->p.counts);
  free(h->h_reward_lut);
  for (int c = 0; c < 16; ++c)
    if (h->chunk_ev[c]) cudaEventDestroy(h->chunk_ev[c]);
  if (h->prof_events) {
    for (cudaEvent_t e : *h->prof_events) cudaEventDestroy(e);
    delete h->prof_events;
  }
  delete h;
  return MG_OK;
}

// NoDeath / ActionBonus / PositionBonus (wrappers.py:68-184, 809-882): parameters of K1, see include/minigrid_b200.h
int mg_set_no_death(mg_env *h, int type_mask, double death_cost) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_set_no_death: NULL handle");
  if (type_mask < 0 || type_mask >= (1 << 11)) return fail(MG_ERR_INVALID_ARG, "mg_set_no_death: type_mask has bits beyond OBJECT_TO_IDX (0..10)");
  if (type_mask & (1 << T_GOAL)) return fail(MG_ERR_INVALID_ARG, "goal cannot be a death cell (wrappers.py:845)");
  if (type_mask && h->host_format == MG_HOST_PACKED)
    return fail(MG_ERR_INVALID_ARG, "mg_set_no_death: the packed host format carries no reward value; use MG_HOST_FULL");
  h->p.no_death_mask = type_mask;
  h->p.death_cost = death_cost;
  return MG_OK;
}
int mg_set_bonus(mg_env *h, int mode) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_set_bonus: NULL handle");
  if (mode < 0 || mode > 2) return fail(MG_ERR_INVALID_ARG, "mg_set_bonus: mode is 0 (none), 1 (ActionBonus) or 2 (PositionBonus)");
  if (mode && h->host_format == MG_HOST_PACKED)
    return fail(MG_ERR_INVALID_ARG, "mg_set_bonus: the packed host format carries no reward value; use MG_HOST_FULL");
  MG_ON_DEVICE(h);
  MG_CUDA(cudaDeviceSynchronize());  // no step of this handle may still be counting
  if (h->p.counts) { MG_CUDA(cudaFree(h->p.counts)); h->p.counts = nullptr; }
  h->p.bonus_mode = 0;
  if (mode) {
    const size_t entries = (size_t)h->p.n_envs * (size_t)h->p.g.W * (size_t)h->p.g.H * (mode == 1 ? 28u : 1u);
    MG_CUDA(cudaMalloc(&h->p.counts, entries * sizeof(uint32_t)));
    MG_CUDA(cudaMemset(h->p.counts, 0, entries * sizeof(uint32_t)));
    MG_CUDA(cudaDeviceSynchronize());
    h->p.bonus_mode = mode;
  }
  return MG_OK;
}

int64_t mg_num_envs(const mg_env *h) { return h ? h->p.n_envs : 0; }
int64_t mg_launch_count(const mg_env *h) { return h ? h->launches : 0; }

// The *_host entry points run on the handle's private stream; everything else runs on the caller's stream. The last
// caller stream is remembered so that the private stream can be ordered after the work already enqueued there.
static void note_stream(mg_env *h, cudaStream_t s) {
  if (s != h->hstream) { h->last_stream = s; h->has_last_stream = 1; }
}
static void order_after_caller(mg_env *h) {
  if (!h->has_last_stream) return;
  if (cudaEventRecord(h->ev_order, h->last_stream) == cudaSuccess) cudaStreamWaitEvent(h->hstream, h->ev_order, 0);
  else cudaGetLastError();  // the caller destroyed that stream: its work has completed
  h->has_last_stream = 0;
}

static int seed_impl(mg_env *h, const uint8_t *mask_dev, const uint64_t *seeds_host, uint64_t base_seed, void *stream) {
  MG_ON_DEVICE(h);
  cudaStream_t s = (cudaStream_t)stream;
  note_stream(h, s);
  if (seeds_host) {
    if (!h->d_seeds) MG_CUDA(cudaMalloc(&h->d_seeds, (size_t)h->p.n_envs * sizeof(uint64_t)));
    MG_CUDA(cudaMemcpyAsync(h->d_seeds, seeds_host, (size_t)h->p.n_envs * sizeof(uint64_t), cudaMemcpyHostToDevice, s));
    MG_CUDA(launch_seed(h->p, mask_dev, h->d_seeds, 0, s));
    MG_CUDA(cudaStreamSynchronize(s));  // seeds_host may be pageable and freed by the caller
  } else {
    MG_CUDA(launch_seed(h->p, mask_dev, nullptr, base_seed, s));
  }
  h->launches += 1;
  return MG_OK;
}

int mg_seed(mg_env *h, const uint64_t *seeds_host, void *stream) {
  if (!h || !seeds_host) return fail(MG_ERR_INVALID_ARG, "mg_seed: NULL argument");
  return seed_impl(h, nullptr, seeds_host, 0, stream);
}

int mg_seed_base(mg_env *h, uint64_t base_seed, void *stream) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_seed_base: NULL handle");
  return seed_impl(h, nullptr, nullptr, base_seed, stream);
}

int mg_seed_masked(mg_env *h, const uint8_t *mask_dev, const uint64_t *seeds_host, uint64_t base_seed, void *stream) {
  if (!h || !mask_dev) return fail(MG_ERR_INVALID_ARG, "mg_seed_masked: NULL argument");
  return seed_impl(h, mask_dev, seeds_host, base_seed, stream);
}

int mg_reset(mg_env *h, uint8_t *obs_dev, int32_t *dir_dev, void *stream) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_reset: NULL handle");
  MG_ON_DEVICE(h);
  cudaStream_t s = (cudaStream_t)stream;
  note_stream(h, s);
  MG_CUDA(launch_reset(h->p, nullptr, obs_dev, dir_dev, s));
  h->launches += 1;
  return MG_OK;
}

int mg_reset_masked(mg_env *h, const uint8_t *mask_dev, uint8_t *obs_dev, int32_t *dir_dev, void *stream) {
  if (!h || !mask_dev) return fail(MG_ERR_INVALID_ARG, "mg_reset_masked: NULL argument");
  MG_ON_DEVICE(h);
  cudaStream_t s = (cudaStream_t)stream;
  note_stream(h, s);
  MG_CUDA(launch_reset(h->p, mask_dev, obs_dev, dir_dev, s));
  h->launches += 1;
  return MG_OK;
}

int mg_step(mg_env *h, const void *actions_dev, int action_dtype, uint8_t *obs_dev, int32_t *dir_dev,
            double *reward_dev, uint8_t *terminated_dev, uint8_t *truncated_dev, void *stream) {
  if (!h || !actions_dev) return fail(MG_ERR_INVALID_ARG, "mg_step: NULL argument");
  if (action_dtype < 0 || action_dtype > 2) return fail(MG_ERR_INVALID_ARG, "mg_step: unknown action dtype");
  MG_ON_DEVICE(h);
  cudaStream_t s = (cudaStream_t)stream;
  note_stream(h, s);
  const Params &p = h->p;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  if (h->profiling) {
    MG_CUDA(cudaEventCreate(&ev0));
    MG_CUDA(cudaEventCreate(&ev1));
    MG_CUDA(cudaEventRecord(ev0, s));
  }
  // one launch: transition + autoreset (either mode) + observation
  MG_CUDA(launch_step(p, h->plan, actions_dev, action_dtype, obs_dev, dir_dev, reward_dev, terminated_dev,
                      truncated_dev, nullptr, (int)(h->launches & 1), s));
  h->launches += 1;
  if (h->profiling) {
    MG_CUDA(cudaEventRecord(ev1, s));
    h->prof_events->push_back(ev0);
    h->prof_events->push_back(ev1);
  }
  return MG_OK;
}

int mg_gen_obs(mg_env *h, uint8_t *obs_dev, int32_t *dir_dev, void *stream) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_gen_obs: NULL handle");
  MG_ON_DEVICE(h);
  note_stream(h, (cudaStream_t)stream);
  MG_CUDA(launch_step(h->p, h->plan, nullptr, MG_ACT_I32, obs_dev, dir_dev, nullptr, nullptr, nullptr, nullptr, 0,
                      (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}

int mg_profile(mg_env *h, int enable) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_profile: NULL handle");
  if (!h->prof_events) h->prof_events = new std::vector<cudaEvent_t>();
  h->profiling = enable ? 1 : 0;
  return MG_OK;
}

int mg_profile_read(mg_env *h, double *total_ms, int64_t *n_launches) {
  if (!h || !total_ms || !n_launches) return fail(MG_ERR_INVALID_ARG, "mg_profile_read: NULL argument");
  *total_ms = 0.0; *n_launches = 0;
  if (!h->prof_events) return MG_OK;
  MG_ON_DEVICE(h);
  std::vector<cudaEvent_t> &ev = *h->prof_events;
  for (size_t i = 0; i + 1 < ev.size(); i += 2) {
    MG_CUDA(cudaEventSynchronize(ev[i + 1]));
    float ms = 0.f;
    MG_CUDA(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
    *total_ms += ms; *n_launches += 1;
    cudaEventDestroy(ev[i]); cudaEventDestroy(ev[i + 1]);
  }
  ev.clear();
  return MG_OK;
}

int mg_full_obs(mg_env *h, uint8_t *out_dev, void *stream) {
  if (!h || !out_dev) return fail(MG_ERR_INVALID_ARG, "mg_full_obs: NULL argument");
  MG_ON_DEVICE(h);
  note_stream(h, (cudaStream_t)stream);
  MG_CUDA(launch_full_obs(h->p, out_dev, 1, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}

// ---- SURVEY 8(f-3): observation wrappers on the device (mg_wrappers.cu) ----
int mg_obs_view(mg_env *h, int view_size, uint8_t *out_dev, void *stream) {
  if (!h || !out_dev) return fail(MG_ERR_INVALID_ARG, "mg_obs_view: NULL argument");
  if (view_size < 3 || view_size > 15 || view_size % 2 == 0)
    return fail(MG_ERR_INVALID_ARG, "mg_obs_view: agent_view_size must be odd and in 3..15 (wrappers.py:650-651)");
  MG_ON_DEVICE(h);
  note_stream(h, (cudaStream_t)stream);
  MG_CUDA(launch_view(h->p, view_size, out_dev, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}
int mg_obs_onehot(mg_env *h, const uint8_t *image_dev, int view_size, uint8_t *out_dev, void *stream) {
  if (!h || !image_dev || !out_dev || view_size < 1) return fail(MG_ERR_INVALID_ARG, "mg_obs_onehot: bad argument");
  MG_ON_DEVICE(h);
  MG_CUDA(launch_onehot(image_dev, out_dev, (long long)h->p.n_envs * view_size * view_size, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}
int mg_obs_flat(mg_env *h, const uint8_t *image_dev, int image_bytes, const uint8_t *mission_dev, int mission_bytes, uint8_t *out_dev,
                void *stream) {
  if (!h || !image_dev || !mission_dev || !out_dev || image_bytes < 1 || mission_bytes < 0)
    return fail(MG_ERR_INVALID_ARG, "mg_obs_flat: bad argument");
  MG_ON_DEVICE(h);
  MG_CUDA(launch_flat(image_dev, mission_dev, out_dev, image_bytes, mission_bytes, h->p.n_envs, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}
int mg_obs_symbolic(mg_env *h, int64_t *out_dev, void *stream) {
  if (!h || !out_dev) return fail(MG_ERR_INVALID_ARG, "mg_obs_symbolic: NULL argument");
  MG_ON_DEVICE(h);
  note_stream(h, (cudaStream_t)stream);
  MG_CUDA(launch_symbolic(h->p, (long long *)out_dev, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}
int mg_obs_rgb_partial(mg_env *h, const uint8_t *image_dev, const uint8_t *tiles_dev, const uint16_t *index_dev, uint8_t *out_dev,
                       void *stream) {
  if (!h || !image_dev || !tiles_dev || !index_dev || !out_dev) return fail(MG_ERR_INVALID_ARG, "mg_obs_rgb_partial: NULL argument");
  MG_ON_DEVICE(h);
  MG_CUDA(launch_rgb_partial(image_dev, tiles_dev, index_dev, out_dev, h->p.n_envs, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}
int mg_obs_rgb_full(mg_env *h, const uint8_t *image_dev, const uint8_t *tiles_dev, const uint16_t *index_dev, uint8_t *out_dev,
                    void *stream) {
  if (!h || !image_dev || !tiles_dev || !index_dev || !out_dev) return fail(MG_ERR_INVALID_ARG, "mg_obs_rgb_full: NULL argument");
  MG_ON_DEVICE(h);
  note_stream(h, (cudaStream_t)stream);
  MG_CUDA(launch_rgb_full(h->p, image_dev, tiles_dev, index_dev, out_dev, (cudaStream_t)stream));
  h->launches += 1;
  return MG_OK;
}

static int ensure_host_path(mg_env *h);

int mg_get_state(mg_env *h, uint8_t *grid_dev, int32_t *agent_dev, uint64_t *rng_dev, uint8_t *pending_dev, void *stream) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_get_state: NULL handle");
  MG_ON_DEVICE(h);
  note_stream(h, (cudaStream_t)stream);
  MG_CUDA(launch_get_state(h->p, grid_dev, agent_dev, rng_dev, pending_dev, (cudaStream_t)stream));
  h->launches += (grid_dev ? 1 : 0) + ((agent_dev || rng_dev || pending_dev) ? 1 : 0);
  return MG_OK;
}

int mg_set_state(mg_env *h, const uint8_t *grid_dev, const int32_t *agent_dev, const uint64_t *rng_dev,
                 const uint8_t *pending_dev, void *stream) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_set_state: NULL handle");
  MG_ON_DEVICE(h);
  cudaStream_t s = (cudaStream_t)stream;
  note_stream(h, s);
  MG_CUDA(launch_set_state(h->p, grid_dev, agent_dev, rng_dev, pending_dev, s));
  h->launches += (grid_dev ? 1 : 0) + ((agent_dev || rng_dev || pending_dev) ? 1 : 0);
  if (agent_dev) {
    // K1 trusts the agent records (window offsets, bit-mask shifts): records that fail the range checks were not
    // stored (k_set_agent) and are reported here; this makes an agent injection synchronous.
    int rc = ensure_host_path(h);
    if (rc != MG_OK) return rc;
    MG_CUDA(cudaMemcpyAsync(h->h_err, h->p.err, sizeof(int), cudaMemcpyDeviceToHost, s));
    MG_CUDA(cudaStreamSynchronize(s));
    if (*h->h_err & ERR_BAD_STATE) {
      MG_CUDA(launch_clear_err(h->p, ERR_BAD_STATE, s));
      return fail(MG_ERR_INVALID_ARG, "mg_set_state: agent record out of range (need 0 <= x < width, 0 <= y < height, "
                                      "0 <= dir <= 3, carry type in {-1, key 5, ball 6, box 7}, colour 0..5, step_count >= 0); "
                                      "such records were left unchanged");
    }
  }
  return MG_OK;
}

static int ensure_host_path(mg_env *h) {
  if (h->h_err) return MG_OK;
  const size_t n = (size_t)h->p.n_envs;
  MG_CUDA(cudaMalloc(&h->d_actions, n * sizeof(int32_t)));
  MG_CUDA(cudaMalloc(&h->d_out, align_up(n * OBS_BYTES, 256) + align_up(n * 8, 256) + align_up(n * 4, 256) + 2 * align_up(n, 256)));
  MG_CUDA(cudaHostAlloc(&h->h_err, sizeof(int), cudaHostAllocDefault));
  return MG_OK;
}

int mg_check_error(mg_env *h, void *stream) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_check_error: NULL handle");
  MG_ON_DEVICE(h);
  cudaStream_t s = (cudaStream_t)stream;
  int rc = ensure_host_path(h);
  if (rc != MG_OK) return rc;
  MG_CUDA(cudaMemcpyAsync(h->h_err, h->p.err, sizeof(int), cudaMemcpyDeviceToHost, s));
  MG_CUDA(cudaStreamSynchronize(s));
  if (*h->h_err & ERR_BAD_ACTION) {
    MG_CUDA(launch_clear_err(h->p, ERR_BAD_ACTION, s));
    return fail(MG_ERR_INVALID_ACTION, "Unknown action: outside 0..6 (minigrid_env.py:584-585)");
  }
  return MG_OK;
}

static bool is_pinned(const void *ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess) { cudaGetLastError(); return false; }
  return a.type == cudaMemoryTypeHost;
}

// D2H of one output array: straight into the caller's buffer when it is page-locked, else through the
// handle's pinned staging (copied out after the stream sync).
struct PendingCopy { void *dst; const void *src; size_t bytes; };

static int host_outputs(mg_env *h, uint8_t *obs_host, int32_t *dir_host, double *reward_host, uint8_t *term_host,
                        uint8_t *trunc_host, uint8_t *d_obs, double *d_rew, int32_t *d_dir, uint8_t *d_term, uint8_t *d_trunc) {
  const size_t n = (size_t)h->p.n_envs;
  cudaStream_t s = h->hstream;
  PendingCopy pend[5];
  int np = 0;
  size_t stage_off = 0;
  auto copy_out = [&](void *host, const void *dev, size_t bytes) -> cudaError_t {
    if (!host) return cudaSuccess;
    if (is_pinned(host)) return cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, s);
    if (!h->h_out) {
      cudaError_t e = cudaHostAlloc(&h->h_out, align_up(n * OBS_BYTES, 256) + align_up(n * 8, 256) + align_up(n * 4, 256) + 2 * align_up(n, 256),
                                    cudaHostAllocDefault);
      if (e != cudaSuccess) return e;
    }
    uint8_t *st = h->h_out + stage_off;
    stage_off += align_up(bytes, 256);
    pend[np++] = PendingCopy{host, st, bytes};
    return cudaMemcpyAsync(st, dev, bytes, cudaMemcpyDeviceToHost, s);
  };
  MG_CUDA(copy_out(obs_host, d_obs, n * OBS_BYTES));
  MG_CUDA(copy_out(reward_host, d_rew, n * 8));
  MG_CUDA(copy_out(dir_host, d_dir, n * 4));
  MG_CUDA(copy_out(term_host, d_term, n));
  MG_CUDA(copy_out(trunc_host, d_trunc, n));
  MG_CUDA(cudaMemcpyAsync(h->h_err, h->p.err, sizeof(int), cudaMemcpyDeviceToHost, s));
  MG_CUDA(cudaStreamSynchronize(s));
  for (int i = 0; i < np; ++i) memcpy(pend[i].dst, pend[i].src, pend[i].bytes);
  if (*h->h_err & ERR_BAD_ACTION) {
    MG_CUDA(launch_clear_err(h->p, ERR_BAD_ACTION, s));
    return fail(MG_ERR_INVALID_ACTION, "Unknown action: outside 0..6 (minigrid_env.py:584-585)");
  }
  return MG_OK;
}

static void host_dev_ptrs(mg_env *h, uint8_t **obs, double **rew, int32_t **dir, uint8_t **term, uint8_t **trunc) {
  const size_t n = (size_t)h->p.n_envs;
  uint8_t *b = h->d_out;
  *obs = b; b += align_up(n * OBS_BYTES, 256);
  *rew = (double *)b; b += align_up(n * 8, 256);
  *dir = (int32_t *)b; b += align_up(n * 4, 256);
  *term = b; b += align_up(n, 256);
  *trunc = b;
}

int mg_set_host_format(mg_env *h, int format, int n_threads) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_set_host_format: NULL handle");
  if (format != MG_HOST_FULL && format != MG_HOST_PACKED) return fail(MG_ERR_INVALID_ARG, "mg_set_host_format: unknown format");
  MG_ON_DEVICE(h);
  if (format == MG_HOST_PACKED && (h->p.no_death_mask || h->p.bonus_mode))
    return fail(MG_ERR_INVALID_ARG, "mg_set_host_format: the packed record carries no reward value, and NoDeath / the bonus wrappers change it");
  if (format == MG_HOST_PACKED) {
    const size_t n_pad = (size_t)h->p.n_tiles * TILE;
    if (!h->d_packed) MG_CUDA(cudaMalloc(&h->d_packed, n_pad * PACKED_BYTES));
    if (!h->h_packed) MG_CUDA(cudaHostAlloc(&h->h_packed, n_pad * PACKED_BYTES, cudaHostAllocDefault));
    int want = n_threads > 0 ? n_threads : usable_host_threads();
    if (want > 64) want = 64;
    if ((int64_t)want * 256 > h->p.n_envs) want = (int)(h->p.n_envs / 256 > 0 ? h->p.n_envs / 256 : 1);  // no point in slices of a few envs
    h->pool_threads = want;
    {
      std::lock_guard<std::mutex> lk(g_pool_mu);
      if (!g_pool || g_pool->threads() != want) {
        delete g_pool;
        g_pool = new HostPool(want);
      }
    }
    // chunks: enough of them that the expansion of chunk c overlaps the copy of chunk c + 1, each still a large copy
    int chunks = (int)(h->p.n_envs / 16384);
    chunks = chunks < 1 ? 1 : (chunks > 8 ? 8 : chunks);
    if (const char *e = getenv("MINIGRID_B200_HOST_CHUNKS")) { chunks = atoi(e); chunks = chunks < 1 ? 1 : (chunks > 16 ? 16 : chunks); }  // tuning knob
    for (int c = 0; c < chunks; ++c)
      if (!h->chunk_ev[c]) MG_CUDA(cudaEventCreateWithFlags(&h->chunk_ev[c], cudaEventDisableTiming));
    h->n_chunks = chunks;
  }
  h->host_format = format;
  return MG_OK;
}
int64_t mg_host_d2h_bytes(const mg_env *h) {
  if (!h) return 0;
  return h->host_format == MG_HOST_PACKED ? (int64_t)h->p.n_envs * PACKED_BYTES : (int64_t)h->p.n_envs * (OBS_BYTES + 4 + 8 + 1 + 1);
}
int mg_host_threads(const mg_env *h) { return (h && h->host_format == MG_HOST_PACKED) ? h->pool_threads : 0; }

// MG_HOST_PACKED step: H2D actions, K1 writing 52-byte records, D2H in chunks; the pool expands chunk c into the
// caller's arrays while chunk c + 1 is still on the bus.
static int step_host_packed(mg_env *h, const int32_t *src, uint8_t *obs_host, int32_t *dir_host, double *reward_host,
                            uint8_t *term_host, uint8_t *trunc_host) {
  const size_t n = (size_t)h->p.n_envs;
  cudaStream_t s = h->hstream;
  std::lock_guard<std::mutex> pool_lock(g_pool_mu);
  if (!g_pool) g_pool = new HostPool(h->pool_threads > 0 ? h->pool_threads : 1);
  HostPool *pool = g_pool;
  ExpandJob job;
  job.packed = h->h_packed; job.max_steps = h->p.max_steps; job.reward_lut = h->h_reward_lut;
  const int64_t cal_pos = h->packed_steps % 8192;  // a calibration opens every 8192 steps
  const bool calibrating = h->stream_fixed < 0 && cal_pos < 20;
  if (h->stream_fixed >= 0) job.stream = h->stream_fixed;
  else if (calibrating) job.stream = cal_pos >= 10;
  else job.stream = h->stream_mode;
  if (calibrating && cal_pos == 0) { h->cal_us[0] = h->cal_us[1] = 0.0; h->cal_n[0] = h->cal_n[1] = 0; }
  job.obs = obs_host; job.dir = dir_host; job.reward = reward_host; job.term = term_host; job.trunc = trunc_host;
  int64_t bounds[17];
  const int C = h->n_chunks;
  // whole tiles, and whole cache lines on the host. Eight chunks are not equal: a small first one (the expansion starts
  // sooner), small last ones (less is left to expand once the bus has gone quiet), the bulk in between
  static const int w8[9] = {0, 1, 3, 6, 9, 12, 14, 15, 16};
  for (int c = 0; c <= C; ++c) bounds[c] = (int64_t)((C == 8 ? n * (size_t)w8[c] / 16 : n * (size_t)c / (size_t)C) / 64 * 64);
  bounds[C] = (int64_t)n;
  const auto t0 = std::chrono::steady_clock::now();
  auto since = [&]() { return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now() - t0).count(); };
  double t_enq = 0, t_first = 0, t_last = 0;
  pool->begin(job, bounds, C);  // the workers wake up while the copy and the kernel run
  cudaError_t e = cudaMemcpyAsync(h->d_actions, src, n * sizeof(int32_t), cudaMemcpyHostToDevice, s);
  if (e == cudaSuccess)
    e = launch_step(h->p, h->plan, h->d_actions, MG_ACT_I32, nullptr, nullptr, nullptr, nullptr, nullptr, h->d_packed, (int)(h->launches & 1), s);
  h->launches += 1;
  for (int c = 0; c < C && e == cudaSuccess; ++c) {
    const size_t off = (size_t)bounds[c] * PACKED_BYTES, len = (size_t)(bounds[c + 1] - bounds[c]) * PACKED_BYTES;
    e = cudaMemcpyAsync(h->h_packed + off, reinterpret_cast<const uint8_t *>(h->d_packed) + off, len, cudaMemcpyDeviceToHost, s);
    if (e == cudaSuccess) e = cudaEventRecord(h->chunk_ev[c], s);
  }
  if (e == cudaSuccess) e = cudaMemcpyAsync(h->h_err, h->p.err, sizeof(int), cudaMemcpyDeviceToHost, s);
  int released = 0;
  t_enq = since();
  for (int c = 0; c < C && e == cudaSuccess; ++c) {
    // poll: a chunk lands every ~30 us, a blocking synchronise would add its wake-up latency to each of them
    while ((e = cudaEventQuery(h->chunk_ev[c])) == cudaErrorNotReady) {}
    if (e == cudaSuccess) { pool->chunk_ready(); ++released; }
    if (c == 0) t_first = since();
  }
  t_last = since();
  if (e != cudaSuccess) pool->abort_chunks(C);  // let the workers run through (their output is discarded by the error)
  (void)released;
  pool->wait();
  if (h->trace) {
    h->tr_enqueue += t_enq; h->tr_first_chunk += t_first; h->tr_last_chunk += t_last; h->tr_pool += since(); h->tr_n += 1;
  }
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  if (h->trace) h->tr_total += since();
  if (calibrating && cal_pos % 10 >= 4) {  // (the first four steps of a block settle the caches)
    h->cal_us[job.stream] += since(); h->cal_n[job.stream] += 1;
    if (cal_pos == 19) {
      h->stream_mode = h->cal_us[1] * h->cal_n[0] < h->cal_us[0] * h->cal_n[1] ? 1 : 0;
      if (h->trace) fprintf(stderr, "[minigrid_b200] host expansion: plain %.1f us, streaming %.1f us per step -> %s stores\n",
                            h->cal_us[0] / h->cal_n[0], h->cal_us[1] / h->cal_n[1], h->stream_mode ? "streaming" : "plain");
    }
  }
  h->packed_steps += 1;
  if (e != cudaSuccess) return fail(MG_ERR_CUDA, std::string("mg_step_host (packed): ") + cudaGetErrorString(e));
  if (*h->h_err & ERR_PACKED_RANGE) {
    MG_CUDA(launch_clear_err(h->p, ERR_PACKED_RANGE, s));
    return fail(MG_ERR_INVALID_ARG, "mg_step_host: a rewarded step count exceeds what the packed record holds (2^19 - 1); use MG_HOST_FULL");
  }
  if (*h->h_err & ERR_BAD_ACTION) {
    MG_CUDA(launch_clear_err(h->p, ERR_BAD_ACTION, s));
    return fail(MG_ERR_INVALID_ACTION, "Unknown action: outside 0..6 (minigrid_env.py:584-585)");
  }
  return MG_OK;
}

int mg_reset_host(mg_env *h, uint8_t *obs_host, int32_t *dir_host) {
  if (!h) return fail(MG_ERR_INVALID_ARG, "mg_reset_host: NULL handle");
  MG_ON_DEVICE(h);
  int rc = ensure_host_path(h);
  if (rc != MG_OK) return rc;
  uint8_t *d_obs, *d_term, *d_trunc; double *d_rew; int32_t *d_dir;
  host_dev_ptrs(h, &d_obs, &d_rew, &d_dir, &d_term, &d_trunc);
  order_after_caller(h);
  rc = mg_reset(h, d_obs, d_dir, h->hstream);
  if (rc != MG_OK) return rc;
  return host_outputs(h, obs_host, dir_host, nullptr, nullptr, nullptr, d_obs, d_rew, d_dir, d_term, d_trunc);
}

int mg_step_host(mg_env *h, const int32_t *actions_host, uint8_t *obs_host, int32_t *dir_host, double *reward_host,
                 uint8_t *terminated_host, uint8_t *truncated_host) {
  if (!h || !actions_host) return fail(MG_ERR_INVALID_ARG, "mg_step_host: NULL argument");
  MG_ON_DEVICE(h);
  int rc = ensure_host_path(h);
  if (rc != MG_OK) return rc;
  const size_t n = (size_t)h->p.n_envs;
  const int32_t *src = actions_host;
  if (!is_pinned(actions_host)) {
    if (!h->h_actions) MG_CUDA(cudaHostAlloc(&h->h_actions, n * sizeof(int32_t), cudaHostAllocDefault));
    memcpy(h->h_actions, actions_host, n * sizeof(int32_t));
    src = h->h_actions;
  }
  order_after_caller(h);
  if (h->host_format == MG_HOST_PACKED)
    return step_host_packed(h, src, obs_host, dir_host, reward_host, terminated_host, truncated_host);
  MG_CUDA(cudaMemcpyAsync(h->d_actions, src, n * sizeof(int32_t), cudaMemcpyHostToDevice, h->hstream));
  uint8_t *d_obs, *d_term, *d_trunc; double *d_rew; int32_t *d_dir;
  host_dev_ptrs(h, &d_obs, &d_rew, &d_dir, &d_term, &d_trunc);
  rc = mg_step(h, h->d_actions, MG_ACT_I32, d_obs, d_dir, d_rew, d_term, d_trunc, h->hstream);
  if (rc != MG_OK) return rc;
  return host_outputs(h, obs_host, dir_host, reward_host, terminated_host, truncated_host, d_obs, d_rew, d_dir, d_term, d_trunc);
}
