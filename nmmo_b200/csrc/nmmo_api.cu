// nmmo_api.cu -- host side of the C ABI (include/nmmo_b200.h): allocation, launches, copies.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>
#include <algorithm>

#include "nmmo_device.cuh"
#include "../../include/nmmo_b200.h"

// unity build: the kernels live in their own files but compile into this translation unit
#include "nmmo_step.cu"
#include "nmmo_obs.cu"
#include "nmmo_rollout.cu"
#include "nmmo_state.cu"
#include "nmmo_events.cu"

static thread_local std::string g_err;
static int fail(int code, const std::string &msg) { g_err = msg; return code; }
#define CU(call)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) return fail(NM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

static size_t a16(size_t x) { return (x + 15) & ~(size_t)15; }

// ---------------------------------------------------------------------------------------------- launch plan ----
// One environment of step_body<V>: its dynamic shared memory and its HBM workspace, array by array in the order of the
// carve there (carve / carve_ws, each array rounded to 16 bytes)
struct NmStepBytes { size_t smem, ws; };
template <class V>
static NmStepBytes step_bytes(const NmParams &p) {
  constexpr size_t kSlack = 128;
  typedef typename V::tile_t tile_t;
  const size_t P = p.P, N = p.N, R = p.R, S = p.S, CAP = p.CAP, NINV = p.cfg[NC_N_INV];
  NmStepBytes b{0, 0};
  auto carve = [&](size_t bytes) { b.smem += a16(bytes); };
  auto carve_ws = [&](size_t bytes, bool in_ws = V::kGlobalTables || V::kScratchInWs) { (in_ws ? b.ws : b.smem) += a16(bytes); };
  if (!V::kGlobalTables) { carve(EA_N * R * 2); if (!V::kItemsInPlace) carve(IS_N * CAP * 2); carve(S * S / 2); }      // ent, item, map
  carve((S * S + 31) / 32 * 4);                                       // occ
  carve((CAP + 31) / 32 * 4); carve((CAP + 31) / 32 * 4);             // used, fresh
  carve_ws(P * NINV * 2, V::kScratchInWs);                            // inv
  carve(P);                                                           // invn
  carve_ws(A_N * P * 2);                                              // act
  carve(N); carve(N * 2);                                             // npc_move, npc_att
  carve_ws((size_t)V::kEvCap * 8, V::kItemsInPlace || V::kGlobalTables || V::kScratchInWs);      // ev
  carve_ws(P * 4, V::kScratchInWs);                                   // duniq
  if (!V::kScratchInWs) carve(P * 4);                                 // s_list
  carve((size_t)V::kNpcHash * 2);                                     // npc_hash
  carve_ws(P * 16); carve_ws(P * 8);                                  // task, acc
  carve(std::max<size_t>(4096, R * 8) + (V::kScratchInWs ? 0 : 32 * V::kChunkIters * 4));      // s_scratch
  carve(R * (sizeof(tile_t) + 2));                                    // s_mv
  if (!V::kGlobalTables && !V::kScratchInWs) carve((size_t)V::kDeplCap * sizeof(tile_t));      // dlist
  if (!V::kScratchInWs) carve((size_t)V::kTblSlots * 4);              // s_tbl
  carve_ws(P, V::kScratchInWs);                                       // slow
  if (!V::kScratchInWs) carve(P * 4);                                 // s_plist
  carve(32 * 4); carve(16);                                           // sc, bar
  b.smem += kSlack;
  if (V::kGlobalTables) b.ws += kSlack;      // (the big family's workspace has the same slack, the small layouts' none)
  return b;
}

// The dynamic shared memory of one obs_body<V> CTA, array by array in the order of the carve there
template <class V>
static size_t obs_bytes(const NmParams &p) {
  constexpr size_t kSlack = V::kStage ? 64 : 128;
  constexpr size_t NW = NM_OBS_THREADS / 32;
  const int AP = V::kStage ? p.P : std::min(p.P, NM_BIG_OBS_AGENTS);
  const size_t R = p.R, S = p.S, A = AP, R32 = (R + 31) & ~(size_t)31, ncx = (S + NM_OBS_CELL - 1) / NM_OBS_CELL;
  size_t s = 0;
  auto carve = [&](size_t bytes) { s += a16(bytes); };
  if (V::kStage) {
    carve(EA_N_OBS * (R + NM_OBS_ENT_SKEW) * 2); carve(R * 2);          // s_ent, s_status
    carve(IS_N * (size_t)p.ICAP * 2); carve(S * S / 2);                 // s_item, s_map
  }
  carve((size_t)p.L.n_mkt * IA_N_OBS * 2); carve((size_t)p.L.n_mkt * 2);      // s_mkt, s_mkt_rows
  carve(A * p.cfg[NC_N_INV] * 2); carve(A * 4); carve(128 * 4);               // s_inv, s_invn, s_scan
  carve(NW * a16((size_t)p.L.n_ent * 2));                                     // s_vis_all
  carve(NW * NM_OBS_BATCH * 33 * 4); carve(NW * NM_OBS_BATCH * 2); carve(NW * NM_OBS_BATCH * AC_N * 2);      // s_bb_all, s_ba_all, s_pick_all
  if (V::kStage) carve(NW * NM_OBS_EROWS * 64);                               // s_ebuf_all
  carve(R32 * 4);                                                             // s_pos
  carve((ncx * ncx + 1) * 4); carve(R32 * 2); carve(NW * (R32 / 32) * 4);     // s_cend, s_crow, s_vbm_all
  carve((3 * AC_N + 2) * 4); carve(A * 8); carve(A * 4); carve(A * 8);        // s_head, s_hash, s_meta, s_work
  if (nm_obs_pre_ok(p.R, AP)) { carve(A * 33 * 2); carve(A * 3 * 4); }        // s_va, s_tg
  carve(16);                                                                  // bar
  return s + kSlack;
}

// Test hooks: environment variables that steer nmmo_create's choices, read when an NmHooks is constructed
struct NmHooks {
  static int num(const char *name, int unset) { const char *v = getenv(name); return v ? atoi(v) : unset; }
  bool force_big = num("NMMO_B200_FORCE_BIG", 0) == 1;       // the big family on a small shape
  int envs_per_cta = num("NMMO_B200_ENVS_PER_CTA", 4);       // 4: four per CTA, else three; >= 3: three; 1: one; else two if they fit
  bool no_std_step = num("NMMO_B200_NO_STD_STEP", 0) == 1;   // the generic step kernel (big family: observation kernel too) ...
  bool no_std_obs = num("NMMO_B200_NO_STD_OBS", 0) == 1;     // ... the generic small observation kernel, on a compile-time shape
  bool no_depl_list = getenv("NMMO_B200_NO_DEPL_LIST") != nullptr;      // never trust the depleted-tile list
  int ev_cap = num("NMMO_B200_EV_CAP", 0);                   // a smaller event ring, to provoke overflow
  int icap = num("NMMO_B200_ICAP", 0);                       // a tiny staged item prefix: the observation kernel's HBM tail path
  int h2d_split_min = num("NMMO_B200_H2D_SPLIT_MIN", 0);     // the smallest handle whose byte-packed actions arrive in two ranges
};

// A kernel instantiation and its name as a profiler lists it
struct NmKernel { void (*fn)(NmParams); const char *name; };
#define NM_KERNEL(k) NmKernel{k, #k}

// How a handle launches its step and observation kernels (plan_launches)
struct NmPlan {
  int big;                       // family (NmParams.big)
  int envs_per_cta, threads_per_env;
  int half_smem;                 // step kernel, per environment: dynamic shared memory (NmParams.half_smem) ...
  size_t ws_bytes;               // ... and HBM workspace (NmParams.ws_bytes; 0 = none)
  size_t obs_smem;               // observation kernel: dynamic shared memory per CTA ...
  int obs_parts;                 // ... and CTAs per environment
  // lean: the *_std instantiation where the handle has its compile-time shape, else the generic one; full: the generic
  // one, the only one with the phase profiler and (step kernels) the injected-draw lookup
  NmKernel step_lean, step_full, obs_lean, obs_full;
};

// The handle's shape is the compile-time shape SH (StdShape, StdShape5): its table shape, the record layout and the
// engine defaults the *_std kernels fold in (nm_cfg_std_value)
template <class SH>
static bool has_std_shape(const NmParams &p) {
  constexpr nm_obs_layout sl = nm_std_layout();
  for (int i = 0; i < NC_COUNT; i++)
    if (nm_cfg_std_value(i) != NM_CFG_RUNTIME && p.cfg[i] != nm_cfg_std_value(i)) return false;
  return memcmp(&p.L, &sl, sizeof(sl)) == 0 && p.P == SH::P && p.N == SH::N && p.R == SH::R && p.S == SH::S && p.CAP == SH::CAP &&
         p.cfg[NC_N_INV] == SH::NINV;
}

// The family, the envs per CTA, the sizes and the kernels of a handle of shape `p` (cfg, L, P, N, R, S, CAP, ICAP) on a
// device with `max_smem` bytes of opt-in shared memory per block.  False: an environment does not fit.  No CUDA calls.
static bool plan_launches(const NmParams &p, int max_smem, const NmHooks &hk, NmPlan &pl) {
  auto r128 = [](size_t x) { return (x + 127) & ~(size_t)127; };
  // Two kernel families (csrc/nmmo_step.cu): environments of up to 256 players / 512 entities / 255^2 tiles run out of
  // shared memory, 256 threads each; larger ones (BASELINE.json configs[4]: 1024 players, 2048 NPCs, 544^2 tiles) keep
  // their tables in HBM / L2 and get 1024 threads
  pl.big = (hk.force_big || p.P > NM_STEP_THREADS || p.R > 2 * NM_STEP_THREADS || p.S > 255) ? 1 : 0;
  const NmStepBytes one = pl.big ? step_bytes<VBig>(p) : step_bytes<VSmall>(p);
  pl.obs_smem = pl.big ? obs_bytes<OBig>(p) : obs_bytes<OSmall>(p);
  if (one.smem > (size_t)max_smem || pl.obs_smem > (size_t)max_smem) return false;
  NmStepBytes b = one;
  bool step_std, obs_std;
  if (pl.big) {
    pl.envs_per_cta = 1; pl.threads_per_env = VBig::kThreads;
    pl.step_full = NM_KERNEL(nmmo_step_big_kernel); pl.step_lean = NM_KERNEL(nmmo_step_big_std_kernel);
    pl.obs_full = NM_KERNEL(nmmo_obs_big_kernel); pl.obs_lean = NM_KERNEL(nmmo_obs_big_std_kernel);
    step_std = obs_std = has_std_shape<StdShape5>(p) && p.cfg[NC_VISION] == StdShape5::VIS && !hk.no_std_step;
  } else {
    // four environments per CTA (VSmall4) when they fit, else three (item table and event ring in place in HBM / L2),
    // else two (they walk the code together), else one
    const NmStepBytes four = step_bytes<VSmall4>(p), three = step_bytes<VSmall3>(p);
    const int want = hk.envs_per_cta;
    if (want == 4 && p.P <= VSmall4::kThreads && p.R <= 2 * VSmall4::kThreads && 4 * r128(four.smem) <= (size_t)max_smem) {
      pl.envs_per_cta = 4; pl.threads_per_env = VSmall4::kThreads; b = four;
      pl.step_full = NM_KERNEL(nmmo_step4_kernel); pl.step_lean = NM_KERNEL(nmmo_step4_std_kernel);
    } else if (want >= 3 && 3 * r128(three.smem) <= (size_t)max_smem) {
      pl.envs_per_cta = 3; pl.threads_per_env = VSmall3::kThreads; b = three;
      pl.step_full = NM_KERNEL(nmmo_step3_kernel); pl.step_lean = NM_KERNEL(nmmo_step3_std_kernel);
    } else {
      pl.envs_per_cta = (want != 1 && 2 * r128(one.smem) <= (size_t)max_smem) ? 2 : 1; pl.threads_per_env = VSmall::kThreads;
      pl.step_full = pl.step_lean = NM_KERNEL(nmmo_step_kernel);
    }
    pl.obs_full = NM_KERNEL(nmmo_obs_kernel); pl.obs_lean = NM_KERNEL(nmmo_obs_std_kernel);
    const bool std_shape = has_std_shape<StdShape>(p);
    step_std = std_shape && !hk.no_std_step;
    obs_std = std_shape && p.ICAP == StdShape::ICAP && p.cfg[NC_VISION] == StdShape::VIS && !hk.no_std_obs;
  }
  if (!step_std) pl.step_lean = pl.step_full;
  if (!obs_std) pl.obs_lean = pl.obs_full;
  pl.half_smem = (int)r128(b.smem); pl.ws_bytes = b.ws;
  pl.obs_parts = pl.big ? (p.P + NM_BIG_OBS_AGENTS - 1) / NM_BIG_OBS_AGENTS : 1;
  return true;
}

// The opt-in limit is a property of the kernel, not of the handle: several handles of different shapes may be alive in
// one process, so it only ever grows (per kernel and device)
static int raise_smem_limit(const NmKernel &k, int device, size_t bytes) {
  static std::map<std::pair<void (*)(NmParams), int>, size_t> limit;
  size_t &cur = limit[{k.fn, device}];
  if (bytes > cur) { CU(cudaFuncSetAttribute(k.fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes)); cur = bytes; }
  return NM_OK;
}

struct nmmo_handle {
  NmParams prm;
  int device;
  cudaStream_t copy_stream = nullptr;      // host-buffer path: results go home underneath the observation kernel
  cudaEvent_t ev_step_done = nullptr, ev_copy_done = nullptr;
  unsigned long long *h_overflow = nullptr;   // pinned: event-ring overflow counter, copied home with the results
  // byte-packed host path: the actions arrive in two env ranges on their own stream; the step kernel of the first range runs
  // underneath the copy of the second
  cudaStream_t h2d_stream = nullptr;
  cudaEvent_t ev_entry = nullptr, ev_h2d[2] = {nullptr, nullptr};
  int h2d_split_min = 1024;                   // handles with fewer environments copy in one piece
  NmPlan plan;                                // kernels and launch shapes (plan_launches)
  std::vector<void *> allocs;
  int32_t *d_actions;             // staging for the host-buffer path
  int16_t *d_actions16;           // ... and for its int16 variant
  // injected rng (host mirror, rebuilt on change)
  std::vector<std::vector<std::pair<uint64_t, uint32_t>>> inj;
  uint64_t *d_inj_keys; uint32_t *d_inj_vals; int32_t *d_inj_off;
  uint8_t *d_env_mask;
  // optional per-kernel timing (CUDA events on the launching stream)
  bool timing = false;
  std::vector<cudaEvent_t> ev;    // triples: before step kernel, between, after obs kernel
  size_t ev_used = 0;
  // environment state blobs (nmmo_state.cu): the section table of this handle's family and shape, with the header
  NmStateArgs state;
  // event log (nmmo_events.cu): first row of each env in its nmmo_events call ([E]; calls over disjoint ranges touch
  // disjoint entries); allocated with the staging
  int32_t *ev_off = nullptr;
};

template <typename T>
static int dalloc(nmmo_handle *h, T **ptr, size_t count, bool zero = true) {
  void *q = nullptr;
  size_t bytes = std::max<size_t>(count * sizeof(T), 16);
  CU(cudaMalloc(&q, bytes));
  if (zero) CU(cudaMemset(q, 0, bytes));
  h->allocs.push_back(q);
  *ptr = (T *)q;
  return 0;
}
#define DA(ptr, count) do { int rc_ = dalloc(h, &(ptr), (count)); if (rc_) return rc_; } while (0)

extern "C" const char *nmmo_last_error(void) { return g_err.c_str(); }

// 64-bit digest of what a handle was created from (everything but n_envs, device and env_base): a state blob means
// nothing under other maps (respawn reads the source map), another task table (task ids index it) or another config
static uint64_t digest_bytes(uint64_t d, const void *data, size_t n) {
  const uint8_t *b = (const uint8_t *)data;
  d = nm_mix64(d ^ (uint64_t)n);
  size_t i = 0;
  for (; i + 8 <= n; i += 8) { uint64_t w; memcpy(&w, b + i, 8); d = nm_mix64(d ^ w); }
  uint64_t w = 0;
  memcpy(&w, b + i, n - i);
  return nm_mix64(d ^ w);
}

// The blob layout (DESIGN.md 2.3): a header, then every per-env buffer that is state, each at a 16-byte-aligned offset.
// It depends on the family and the shape only, not on E, env_base, envs per CTA or the std / generic kernel choice.
static void state_layout(nmmo_handle *h, uint64_t digest) {
  NmParams &p = h->prm;
  NmStateArgs &a = h->state;
  memset(&a, 0, sizeof(a));
  uint32_t off = NM_STATE_HEADER;
  auto add = [&](void *base, size_t h_env, size_t bytes, int live_sc = -1, int unit = 1) {
    NmStateSec &q = a.sec[a.n_sec++];
    q.h = (uint8_t *)base; q.h_env = (uint32_t)h_env; q.b_off = off; q.bytes = (uint32_t)bytes;
    q.live_sc = (int16_t)live_sc; q.unit = (int16_t)unit;
    off = (uint32_t)a16(off + bytes);
  };
  const size_t P = p.P, ent_bytes = (p.big ? (size_t)NM_BIG_ENT_STRIDE : (size_t)EA_N) * p.R * 2;
  const size_t tile = p.big ? sizeof(VBig::tile_t) : sizeof(VSmall::tile_t), depl_cap = p.big ? VBig::kDeplCap : VSmall::kDeplCap;
  a.sc_off = off;
  add(p.scalars, NM_SC_N * 4, NM_SC_N * 4);
  add(p.seed, 8, 8);
  add(p.episode_done, 1, 1);
  add(p.ent, ent_bytes, ent_bytes);
  for (int k = 0; k < IS_N; k++) add(p.item + (size_t)k * p.CAP, (size_t)IS_N * p.CAP * 2, (size_t)p.CAP * 2, SC_ITEM_HI, 2);
  add(p.map, (size_t)p.S * p.S / 2, (size_t)p.S * p.S / 2);
  add(p.depl, depl_cap * tile, depl_cap * tile, SC_N_DEPL, (int)tile);
  add(p.danger, (size_t)p.N * 2, (size_t)p.N * 2, SC_N_DANGER, 2);
  add(p.stats, P * ST_N * 4, P * ST_N * 4);
  add(p.dstats, P * DS_N * 8, P * DS_N * 8);
  add(p.uniq, P * NM_UNIQ_WORDS * 4, P * NM_UNIQ_WORDS * 4);
  add(p.task_id, P * 4, P * 4);
  add(p.rew, P * 4, P * 4);
  add(p.term, P, P); add(p.trunc, P, P); add(p.mask, P, P); add(p.info_valid, P, P);
  add(p.info, P * IN_N * 4, P * IN_N * 4);
  a.state_bytes = (off + 127) & ~127u;
  for (int s = 0; s < a.n_sec; s++) a.sec[s].span = (s + 1 < a.n_sec ? a.sec[s + 1].b_off : a.state_bytes) - a.sec[s].b_off;
  a.n_chunks = (a.state_bytes + NM_STATE_CHUNK - 1) / NM_STATE_CHUNK;
  a.scalars = p.scalars; a.obs_meta = p.obs_meta; a.P = p.P;
  a.hdr.magic = NM_STATE_MAGIC; a.hdr.version = NM_STATE_VERSION; a.hdr.family = (uint32_t)p.big;
  a.hdr.state_bytes = a.state_bytes; a.hdr.digest = digest;
}
static_assert(IS_N + 17 <= NM_STATE_MAX_SECS, "state sections");
static_assert(sizeof(NmStateArgs) <= 4096, "the section table and the env ids travel as kernel parameters");

extern "C" int nmmo_create(const int32_t *cfg, int n_cfg, const double *fcfg, int n_fcfg, int n_envs, int device,
                           int env_base, const uint8_t *maps, int n_maps, const int32_t *tasks,
                           const uint16_t *task_embed, int n_tasks, nmmo_handle **out) {
  if (!cfg || !fcfg || !maps || !tasks || !task_embed || !out) return fail(NM_ERR_ARG, "null argument");
  if (n_cfg != NC_COUNT || n_fcfg != NF_COUNT) return fail(NM_ERR_ARG, "config vector length does not match nmmo_spec.h");
  if (n_envs <= 0 || n_maps <= 0 || n_tasks <= 0) return fail(NM_ERR_ARG, "n_envs, n_maps, n_tasks must be positive");
  if (cfg[NC_DEATH_FOG] < -1 || cfg[NC_DEATH_FOG_SPEED] < 0 || cfg[NC_DEATH_FOG_FINAL_SIZE] < 0)
    return fail(NM_ERR_ARG, "DEATH_FOG must be -1 (off) or a tick >= 0; DEATH_FOG_SPEED and DEATH_FOG_FINAL_SIZE must be >= 0");
  const NmHooks hk{};
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail(NM_ERR_CUDA, "no CUDA device: nmmo_b200 has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(NM_ERR_ARG, "bad device index");
  CU(cudaSetDevice(device));
  nmmo_handle *h = new nmmo_handle();
  struct Guard {      // any early return below frees what was allocated so far
    nmmo_handle *h; bool armed = true;
    ~Guard() { if (armed) { for (void *q : h->allocs) cudaFree(q); delete h; } }
  } guard{h};
  h->device = device;
  NmParams &p = h->prm;
  memset(&p, 0, sizeof(p));
  memcpy(p.cfg, cfg, sizeof(int32_t) * NC_COUNT);
  memcpy(p.fcfg, fcfg, sizeof(double) * NF_COUNT);
  nm_obs_layout_init(p.cfg, &p.L);
  p.E = n_envs; p.P = cfg[NC_N_PLAYERS]; p.N = cfg[NC_N_NPCS]; p.R = p.P + p.N; p.S = cfg[NC_MAP_SIZE]; p.CAP = cfg[NC_ITEM_CAP];
  p.n_maps = n_maps; p.n_tasks = n_tasks; p.env_base = env_base;
  p.ICAP = std::min(p.CAP, 256);      // item rows the observation kernel keeps in shared memory; rows beyond are read in HBM
  if (hk.icap >= 8 && hk.icap % 8 == 0) p.ICAP = std::min(p.CAP, hk.icap);
  if (p.P <= 0 || p.P > NM_BIG_THREADS) { return fail(NM_ERR_LIMIT, "PLAYER_N must be in 1..1024"); }
  if (p.R % 8 || p.CAP % 8 || (p.S * p.S) % 32) { return fail(NM_ERR_LIMIT, "P+N and item cap must be multiples of 8, S*S of 32 (bulk copies)"); }
  if (p.R > VBig::kRowsPerThread * NM_BIG_THREADS) { return fail(NM_ERR_LIMIT, "P+N must be <= 3072"); }
  if (p.S > 1023) { return fail(NM_ERR_LIMIT, "MAP_SIZE must be <= 1023"); }
  if (p.N > VBig::kNpcHash / 2) { return fail(NM_ERR_LIMIT, "NPC_N must be <= 2048"); }
  if (p.cfg[NC_NPC_SPAWN_ATTEMPTS] > 32) { return fail(NM_ERR_LIMIT, "NPC_SPAWN_ATTEMPTS must be <= 32"); }
  if (p.L.n_ent > 255 || p.cfg[NC_N_INV] > 16) { return fail(NM_ERR_LIMIT, "N_ENT_OBS <= 255, N_INV <= 16"); }
  if (p.L.m_end > 1024) { return fail(NM_ERR_LIMIT, "the ActionTargets masks must total <= 1024 entries (one 32-entry word per lane)"); }
  if (p.cfg[NC_SPAWN_PATCH] > 0 && (p.cfg[NC_SPAWN_PATCH] * p.cfg[NC_SPAWN_PATCH] < p.P || p.cfg[NC_SPAWN_PATCH] > p.cfg[NC_MAP_CENTER]))
    return fail(NM_ERR_ARG, "SPAWN_PATCH^2 must hold PLAYER_N players and fit inside the map centre");
  if (p.cfg[NC_SPAWN_PATCH] == 0 && !p.cfg[NC_ALLOW_OCCUPIED] && p.P > 4 * p.cfg[NC_MAP_CENTER])
    return fail(NM_ERR_ARG, "border-ring spawn with one entity per tile needs PLAYER_N <= 4 * MAP_CENTER");
  int max_smem = 0;
  CU(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  NmPlan &pl = h->plan;
  if (!plan_launches(p, max_smem, hk, pl)) { return fail(NM_ERR_LIMIT, "environment does not fit in shared memory"); }
  p.big = pl.big; p.envs_per_cta = pl.envs_per_cta; p.half_smem = pl.half_smem; p.ws_bytes = pl.ws_bytes;
  for (const NmKernel *k : {&pl.step_lean, &pl.step_full}) { int rc = raise_smem_limit(*k, device, (size_t)pl.envs_per_cta * pl.half_smem); if (rc) return rc; }
  for (const NmKernel *k : {&pl.obs_lean, &pl.obs_full}) { int rc = raise_smem_limit(*k, device, pl.obs_smem); if (rc) return rc; }
  p.no_depl_list = hk.no_depl_list;
  p.ev_cap = p.big ? VBig::kEvCap : VSmall::kEvCap;
  if (hk.ev_cap > 0 && hk.ev_cap < p.ev_cap) p.ev_cap = hk.ev_cap;
  size_t E = p.E, P = p.P;
  const size_t ent_i16 = p.big ? (size_t)NM_BIG_ENT_STRIDE * p.R : (size_t)EA_N * p.R;      // int16 per env
  DA(p.ent, E * ent_i16); DA(p.item, E * IS_N * p.CAP); DA(p.map, E * p.S * p.S / 2);
  if (p.ws_bytes) DA(p.ws, E * p.ws_bytes);
  uint8_t *dmaps; DA(dmaps, (size_t)n_maps * p.S * p.S); p.maps = dmaps;
  CU(cudaMemcpy(dmaps, maps, (size_t)n_maps * p.S * p.S, cudaMemcpyHostToDevice));
  DA(p.scalars, E * NM_SC_N); DA(p.seed, E); DA(p.danger, E * p.N);
  { uint8_t *dl; DA(dl, p.big ? E * VBig::kDeplCap * sizeof(VBig::tile_t) : E * VSmall::kDeplCap * sizeof(VSmall::tile_t)); p.depl = dl; }
  DA(p.stats, E * P * ST_N); DA(p.dstats, E * P * DS_N); DA(p.uniq, E * P * NM_UNIQ_WORDS); DA(p.task_id, E * P);
  int32_t *dtasks; DA(dtasks, (size_t)n_tasks * NM_TASK_COLS); p.tasks = dtasks;
  CU(cudaMemcpy(dtasks, tasks, sizeof(int32_t) * n_tasks * NM_TASK_COLS, cudaMemcpyHostToDevice));
  uint16_t *demb; DA(demb, (size_t)n_tasks * p.L.task_dim); p.embed = demb;
  CU(cudaMemcpy(demb, task_embed, sizeof(uint16_t) * n_tasks * p.L.task_dim, cudaMemcpyHostToDevice));
  DA(p.obs, E * P * p.L.stride);
  DA(p.rew, E * P); DA(p.term, E * P); DA(p.trunc, E * P); DA(p.mask, E * P);
  DA(p.info, E * P * IN_N); DA(p.info_valid, E * P); DA(p.episode_done, E);
  DA(p.agg, (size_t)NM_AGG_REP * 2 * IN_N); DA(p.counters, 8); DA(p.obs_meta, E * P);
  DA(h->d_actions, E * P * AC_N);
  DA(h->d_actions16, E * P * AC_N);
  DA(h->d_inj_off, E + 1);
  DA(h->d_env_mask, E);
  h->d_inj_keys = nullptr; h->d_inj_vals = nullptr;
  p.inj_off = nullptr; p.inj_keys = nullptr; p.inj_vals = nullptr;
  h->inj.resize(E);
  // every env starts "done" so that a step before any reset resets from seed 0
  std::vector<int32_t> sc(E * NM_SC_N, 0);
  for (size_t e = 0; e < E; e++) sc[e * NM_SC_N + SC_DONE] = 1;
  CU(cudaMemcpy(p.scalars, sc.data(), sizeof(int32_t) * sc.size(), cudaMemcpyHostToDevice));
  if (hk.h2d_split_min >= 1) h->h2d_split_min = hk.h2d_split_min;
  {
    uint64_t d = 0x6E6D6D6F53544154ULL;
    d = digest_bytes(d, cfg, sizeof(int32_t) * NC_COUNT);
    d = digest_bytes(d, fcfg, sizeof(double) * NF_COUNT);
    d = digest_bytes(d, maps, (size_t)n_maps * p.S * p.S);
    d = digest_bytes(d, tasks, sizeof(int32_t) * n_tasks * NM_TASK_COLS);
    d = digest_bytes(d, task_embed, sizeof(uint16_t) * n_tasks * p.L.task_dim);
    state_layout(h, d);
  }
  guard.armed = false;
  *out = h;
  return NM_OK;
}

extern "C" int nmmo_destroy(nmmo_handle *h) {
  if (!h) return NM_OK;
  cudaSetDevice(h->device);
  cudaDeviceSynchronize();
  for (void *q : h->allocs) cudaFree(q);
  if (h->d_inj_keys) cudaFree(h->d_inj_keys);
  if (h->d_inj_vals) cudaFree(h->d_inj_vals);
  for (cudaEvent_t e : h->ev) cudaEventDestroy(e);
  if (h->h2d_stream) { cudaStreamDestroy(h->h2d_stream); cudaEventDestroy(h->ev_entry); cudaEventDestroy(h->ev_h2d[0]); cudaEventDestroy(h->ev_h2d[1]); }
  if (h->copy_stream) { cudaStreamDestroy(h->copy_stream); cudaEventDestroy(h->ev_step_done); cudaEventDestroy(h->ev_copy_done); cudaFreeHost(h->h_overflow); }
  if (h->prm.ev_log) { cudaFree(h->prm.ev_log); cudaFree(h->prm.ev_n); cudaFree(h->ev_off); }
  if (h->prm.next_flags) { cudaFree(h->prm.next_flags); cudaFree(h->prm.next_seed); cudaFree(h->prm.next_map); cudaFree(h->prm.next_task); }
  delete h;
  return NM_OK;
}

// The plan entry a launch with `prm` uses: the *_std instantiations have no phase profiler and (step kernels) no
// injected-draw lookup
static bool lean(const NmParams &prm, bool step) { return !prm.prof && !(step && prm.inj_off); }
static const NmKernel &step_kernel(const nmmo_handle *h, const NmParams &prm) { return lean(prm, true) ? h->plan.step_lean : h->plan.step_full; }
static const NmKernel &obs_kernel(const nmmo_handle *h, const NmParams &prm) { return lean(prm, false) ? h->plan.obs_lean : h->plan.obs_full; }

// step kernel over env range [lo, hi) on `st`
static int launch_step_kernel(nmmo_handle *h, NmParams &prm, cudaStream_t st, int lo, int hi) {
  const NmPlan &pl = h->plan;
  prm.env_lo = lo; prm.env_hi = hi;
  const auto fn = step_kernel(h, prm).fn;
  fn<<<(hi - lo + pl.envs_per_cta - 1) / pl.envs_per_cta, pl.envs_per_cta * pl.threads_per_env, (size_t)pl.envs_per_cta * pl.half_smem, st>>>(prm);
  CU(cudaGetLastError());
  return NM_OK;
}

// observation kernel over env range [lo, hi) on `st`
static int launch_obs_kernel(nmmo_handle *h, NmParams &prm, cudaStream_t st, int lo, int hi) {
  const NmPlan &pl = h->plan;
  prm.env_lo = lo; prm.env_hi = hi;
  const auto fn = obs_kernel(h, prm).fn;
  fn<<<(hi - lo) * pl.obs_parts, NM_OBS_THREADS, pl.obs_smem, st>>>(prm);
  CU(cudaGetLastError());
  return NM_OK;
}

// step_done = true: the step kernel of this tick was already launched (in env ranges, by the caller)
static int launch_step(nmmo_handle *h, int mode, cudaStream_t st, cudaEvent_t after_step = nullptr, bool step_done = false) {
  NmParams prm = h->prm;
  prm.mode = mode;
  cudaEvent_t *e3 = nullptr;
  if (h->timing && mode == 0) {
    if (h->ev_used + 3 > h->ev.size()) {
      for (int i = 0; i < 3; i++) { cudaEvent_t e; CU(cudaEventCreate(&e)); h->ev.push_back(e); }
    }
    e3 = &h->ev[h->ev_used];
    h->ev_used += 3;
    CU(cudaEventRecord(e3[0], st));
  }
  if (!step_done) { int rc = launch_step_kernel(h, prm, st, 0, prm.E); if (rc) return rc; }
  if (e3) CU(cudaEventRecord(e3[1], st));
  if (after_step) CU(cudaEventRecord(after_step, st));      // rewards / flags / mask are final here
  { int rc = launch_obs_kernel(h, prm, st, 0, prm.E); if (rc) return rc; }
  if (e3) CU(cudaEventRecord(e3[2], st));
  return NM_OK;
}

extern "C" int nmmo_reset(nmmo_handle *h, const uint64_t *seeds, const int32_t *map_ids, const int32_t *task_ids,
                          const uint8_t *env_mask, void *stream) {
  if (!h || !seeds) return fail(NM_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  NmParams &p = h->prm;
  size_t E = p.E, P = p.P;
  // validate everything before any device state is touched: an NM_ERR_ARG return leaves the handle as it was
  for (size_t e = 0; e < E; e++) {
    if (env_mask && !env_mask[e]) continue;
    if (map_ids && (map_ids[e] < 0 || map_ids[e] >= p.n_maps)) return fail(NM_ERR_ARG, "map id out of range");
    if (task_ids)
      for (size_t a = 0; a < P; a++)
        if (task_ids[e * P + a] < 0 || task_ids[e * P + a] >= p.n_tasks) return fail(NM_ERR_ARG, "task id out of range");
  }
  CU(cudaStreamSynchronize(st));
  std::vector<int32_t> sc(E * NM_SC_N);
  CU(cudaMemcpy(sc.data(), p.scalars, sizeof(int32_t) * sc.size(), cudaMemcpyDeviceToHost));
  std::vector<uint64_t> sd(E);
  CU(cudaMemcpy(sd.data(), p.seed, sizeof(uint64_t) * E, cudaMemcpyDeviceToHost));
  for (size_t e = 0; e < E; e++) {
    if (env_mask && !env_mask[e]) continue;
    int32_t *s = &sc[e * NM_SC_N];
    s[SC_NEED_RESET] = 1; s[SC_EPISODE] = 0; s[SC_ERROR] = 0;
    s[SC_EXPLICIT_MAP] = map_ids ? 1 : 0;
    if (map_ids) s[SC_MAP_ID] = map_ids[e];
    s[SC_EXPLICIT_TASKS] = task_ids ? 1 : 0;
    sd[e] = seeds[e];
  }
  // uploads are stream-ordered on `st` with the reset launch below (the host vectors outlive the final synchronize)
  CU(cudaMemcpyAsync(p.scalars, sc.data(), sizeof(int32_t) * sc.size(), cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(p.seed, sd.data(), sizeof(uint64_t) * E, cudaMemcpyHostToDevice, st));
  if (task_ids) {
    for (size_t e = 0; e < E; e++) {
      if (env_mask && !env_mask[e]) continue;
      CU(cudaMemcpyAsync(p.task_id + e * P, task_ids + e * P, sizeof(int32_t) * P, cudaMemcpyHostToDevice, st));
    }
  }
  int rc = launch_step(h, 1, st);
  if (rc) return rc;
  CU(cudaStreamSynchronize(st));
  return NM_OK;
}

extern "C" int nmmo_step(nmmo_handle *h, const int32_t *actions_dev, void *stream) {
  if (!h || !actions_dev) return fail(NM_ERR_ARG, "null argument");
  if ((uintptr_t)actions_dev & 15) return fail(NM_ERR_ARG, "actions must be 16-byte aligned");
  CU(cudaSetDevice(h->device));
  h->prm.actions = actions_dev;
  return launch_step(h, 0, (cudaStream_t)stream);
}

extern "C" int nmmo_step_envs(nmmo_handle *h, int env_lo, int env_hi, const int32_t *actions_dev, void *stream) {
  if (!h || !actions_dev) return fail(NM_ERR_ARG, "null argument");
  if (env_lo < 0 || env_hi > h->prm.E || env_lo >= env_hi) return fail(NM_ERR_ARG, "env range must satisfy 0 <= env_lo < env_hi <= E");
  if ((uintptr_t)actions_dev & 15) return fail(NM_ERR_ARG, "actions must be 16-byte aligned");
  if (h->timing || h->prm.prof)
    return fail(NM_ERR_STATE, "per-kernel timing and the phase profiler describe whole-handle launches: switch them off for range steps");
  CU(cudaSetDevice(h->device));
  NmParams prm = h->prm;
  prm.mode = 0;
  prm.actions = actions_dev; prm.act_env_lo = env_lo;
  const cudaStream_t st = (cudaStream_t)stream;
  int rc = launch_step_kernel(h, prm, st, env_lo, env_hi);
  if (rc) return rc;
  return launch_obs_kernel(h, prm, st, env_lo, env_hi);
}

static int finish_step_host(nmmo_handle *h, float *rew_out, uint8_t *term_out, uint8_t *trunc_out, uint8_t *mask_out,
                            uint8_t *obs_out, cudaStream_t st, bool step_done = false);

extern "C" int nmmo_step_host(nmmo_handle *h, const int32_t *actions_host, float *rew_out, uint8_t *term_out,
                              uint8_t *trunc_out, uint8_t *mask_out, uint8_t *obs_out, void *stream) {
  if (!h || !actions_host) return fail(NM_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  NmParams &p = h->prm;
  size_t n = (size_t)p.E * p.P;
  // the caller's buffers are used directly (pinned memory makes the copies asynchronous)
  CU(cudaMemcpyAsync(h->d_actions, actions_host, n * AC_N * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  return finish_step_host(h, rew_out, term_out, trunc_out, mask_out, obs_out, st);
}

__global__ void nmmo_widen_actions_kernel(const int16_t *src, int32_t *dst, size_t n8) {
  // 8 actions per thread: one 16-byte load, two 16-byte stores
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n8; i += (size_t)gridDim.x * blockDim.x) {
    const uint4 v = ((const uint4 *)src)[i];
    const uint32_t w[4] = {v.x, v.y, v.z, v.w};
    int4 lo, hi;
    lo.x = (int16_t)(w[0] & 0xffffu); lo.y = (int16_t)(w[0] >> 16); lo.z = (int16_t)(w[1] & 0xffffu); lo.w = (int16_t)(w[1] >> 16);
    hi.x = (int16_t)(w[2] & 0xffffu); hi.y = (int16_t)(w[2] >> 16); hi.z = (int16_t)(w[3] & 0xffffu); hi.w = (int16_t)(w[3] >> 16);
    ((int4 *)dst)[2 * i] = lo; ((int4 *)dst)[2 * i + 1] = hi;
  }
}

static int finish_step_host(nmmo_handle *h, float *rew_out, uint8_t *term_out, uint8_t *trunc_out, uint8_t *mask_out,
                            uint8_t *obs_out, cudaStream_t st, bool step_done) {
  NmParams &p = h->prm;
  size_t n = (size_t)p.E * p.P;
  p.actions = h->d_actions;
  // The step kernel writes reward / terminated / truncated / mask; the observation kernel only reads them.
  // Their way back to the host therefore runs on a side stream underneath the observation kernel.
  if (!h->copy_stream) {
    CU(cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&h->ev_step_done, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&h->ev_copy_done, cudaEventDisableTiming));
    CU(cudaMallocHost((void **)&h->h_overflow, sizeof(unsigned long long)));
    *h->h_overflow = 0;
  }
  int rc = launch_step(h, 0, st, h->ev_step_done, step_done);
  if (rc) return rc;
  cudaStream_t cs = h->copy_stream;
  CU(cudaStreamWaitEvent(cs, h->ev_step_done, 0));
  if (rew_out) CU(cudaMemcpyAsync(rew_out, p.rew, n * sizeof(float), cudaMemcpyDeviceToHost, cs));
  if (term_out) CU(cudaMemcpyAsync(term_out, p.term, n, cudaMemcpyDeviceToHost, cs));
  if (trunc_out) CU(cudaMemcpyAsync(trunc_out, p.trunc, n, cudaMemcpyDeviceToHost, cs));
  if (mask_out) CU(cudaMemcpyAsync(mask_out, p.mask, n, cudaMemcpyDeviceToHost, cs));
  CU(cudaMemcpyAsync(h->h_overflow, p.counters + 3, sizeof(unsigned long long), cudaMemcpyDeviceToHost, cs));
  CU(cudaEventRecord(h->ev_copy_done, cs));
  if (obs_out) CU(cudaMemcpyAsync(obs_out, p.obs, n * p.L.stride, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamWaitEvent(st, h->ev_copy_done, 0));
  CU(cudaStreamSynchronize(st));
  if (*h->h_overflow)      // events were dropped: the episode statistics and event-driven task progress of that env are wrong
    return fail(NM_ERR_STATE, "event ring overflow in " + std::to_string(*h->h_overflow) + " env-tick(s): more events in one tick than the ring holds");
  return NM_OK;
}

// Device-side error state (synchronises): NM_ERR_STATE when any environment dropped events (its SC_ERROR bit is set), or an
// automatic reset rejected an out-of-range pending next-episode entry, since the counters were last cleared.  The asynchronous nmmo_step cannot report it; callers poll this at their
// logging cadence (B200VecEnv.stats does).
extern "C" int nmmo_check(nmmo_handle *h) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  unsigned long long n[3] = {0, 0, 0};
  CU(cudaMemcpy(n, h->prm.counters + 3, sizeof(n), cudaMemcpyDeviceToHost));
  if (n[0]) return fail(NM_ERR_STATE, "event ring overflow in " + std::to_string(n[0]) + " env-tick(s): more events in one tick than the ring holds");
  if (n[2])
    return fail(NM_ERR_STATE, std::to_string(n[2]) + " pending next-episode entr" + (n[2] == 1 ? "y was" : "ies were") +
                              " out of range (a next_map id outside [0, " + std::to_string(h->prm.n_maps) + ") or a team's next_task row outside [0, " +
                              std::to_string(h->prm.n_tasks) + ")): automatic resets drew those fields as if they were unset");
  return NM_OK;
}

extern "C" int nmmo_step_host_i16(nmmo_handle *h, const int16_t *actions_host, float *rew_out, uint8_t *term_out,
                                  uint8_t *trunc_out, uint8_t *mask_out, uint8_t *obs_out, void *stream) {
  if (!h || !actions_host) return fail(NM_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t n12 = (size_t)h->prm.E * h->prm.P * AC_N;
  CU(cudaMemcpyAsync(h->d_actions16, actions_host, n12 * sizeof(int16_t), cudaMemcpyHostToDevice, st));
  size_t n8 = n12 / 8;      // P * 12 is a multiple of 8 for every supported P (P+N and the item cap are)
  if (n12 % 8) return fail(NM_ERR_LIMIT, "E * P * 12 must be a multiple of 8 for the int16 action path");
  nmmo_widen_actions_kernel<<<(unsigned)std::min<size_t>((n8 + 255) / 256, 148 * 8), 256, 0, st>>>(h->d_actions16, h->d_actions, n8);
  CU(cudaGetLastError());
  return finish_step_host(h, rew_out, term_out, trunc_out, mask_out, obs_out, st);
}

__global__ void nmmo_unpack_actions_u8_kernel(const uint32_t *src, int4 *dst, size_t n_agents) {
  // one agent per thread: 12 bytes in, 12 int32 out; bits 2..7 of byte 0 are bits 8.. of head 2 (Buy.MarketItem)
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n_agents; i += (size_t)gridDim.x * blockDim.x) {
    const uint32_t a = src[3 * i], b = src[3 * i + 1], c2 = src[3 * i + 2];
    const int b0 = (int)(a & 0xffu);
    dst[3 * i] = make_int4(b0 & 3, (int)((a >> 8) & 0xffu), (int)((a >> 16) & 0xffu) | ((b0 >> 2) << 8), (int)(a >> 24));
    dst[3 * i + 1] = make_int4((int)(b & 0xffu), (int)((b >> 8) & 0xffu), (int)((b >> 16) & 0xffu), (int)(b >> 24));
    dst[3 * i + 2] = make_int4((int)(c2 & 0xffu), (int)((c2 >> 8) & 0xffu), (int)((c2 >> 16) & 0xffu), (int)(c2 >> 24));
  }
}

extern "C" int nmmo_step_host_u8(nmmo_handle *h, const uint8_t *actions_host, float *rew_out, uint8_t *term_out,
                                 uint8_t *trunc_out, uint8_t *mask_out, uint8_t *obs_out, void *stream) {
  if (!h || !actions_host) return fail(NM_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->device));
  cudaStream_t st = (cudaStream_t)stream;
  const nm_obs_layout &L = h->prm.L;
  if (L.n_ent + 1 > 256 || L.n_price > 256 || L.n_inv + 1 > 256 || L.n_mkt + 1 > (1 << 14))
    return fail(NM_ERR_LIMIT, "an action head is too wide for the packed byte format");
  const size_t P = h->prm.P, n = (size_t)h->prm.E * P;
  const int E = h->prm.E, epc = h->prm.envs_per_cta;
  // Large handles: the actions arrive as two env ranges (a quarter, then the rest) on a copy stream, and the step kernel of
  // the first range runs underneath the copy of the second, so only a quarter of the H2D time is exposed.  (Per-kernel
  // timing and profiling want one step launch per tick: they take the one-piece path.)
  const int lo1 = (E / 4) / epc * epc;
  if (E >= h->h2d_split_min && lo1 > 0 && lo1 < E && !h->timing && !h->prm.prof) {
    if (!h->h2d_stream) {
      CU(cudaStreamCreateWithFlags(&h->h2d_stream, cudaStreamNonBlocking));
      CU(cudaEventCreateWithFlags(&h->ev_entry, cudaEventDisableTiming));
      for (int k = 0; k < 2; k++) CU(cudaEventCreateWithFlags(&h->ev_h2d[k], cudaEventDisableTiming));
    }
    CU(cudaEventRecord(h->ev_entry, st));                      // the copies follow whatever the caller queued on `st`
    CU(cudaStreamWaitEvent(h->h2d_stream, h->ev_entry, 0));
    const int cut[3] = {0, lo1, E};
    uint8_t *d16 = (uint8_t *)h->d_actions16;
    for (int k = 0; k < 2; k++) {
      const size_t a0 = (size_t)cut[k] * P, na = (size_t)(cut[k + 1] - cut[k]) * P;
      CU(cudaMemcpyAsync(d16 + a0 * AC_N, actions_host + a0 * AC_N, na * AC_N, cudaMemcpyHostToDevice, h->h2d_stream));
      CU(cudaEventRecord(h->ev_h2d[k], h->h2d_stream));
    }
    h->prm.actions = h->d_actions;
    NmParams prm = h->prm;
    prm.mode = 0;
    for (int k = 0; k < 2; k++) {
      const size_t a0 = (size_t)cut[k] * P, na = (size_t)(cut[k + 1] - cut[k]) * P;
      CU(cudaStreamWaitEvent(st, h->ev_h2d[k], 0));
      nmmo_unpack_actions_u8_kernel<<<(unsigned)std::min<size_t>((na + 255) / 256, 148 * 8), 256, 0, st>>>(
          (const uint32_t *)(d16 + a0 * AC_N), (int4 *)(h->d_actions + a0 * AC_N), na);
      CU(cudaGetLastError());
      int rc = launch_step_kernel(h, prm, st, cut[k], cut[k + 1]);
      if (rc) return rc;
    }
    return finish_step_host(h, rew_out, term_out, trunc_out, mask_out, obs_out, st, true);
  }
  CU(cudaMemcpyAsync(h->d_actions16, actions_host, n * AC_N, cudaMemcpyHostToDevice, st));
  nmmo_unpack_actions_u8_kernel<<<(unsigned)std::min<size_t>((n + 255) / 256, 148 * 8), 256, 0, st>>>(
      (const uint32_t *)h->d_actions16, (int4 *)h->d_actions, n);
  CU(cudaGetLastError());
  return finish_step_host(h, rew_out, term_out, trunc_out, mask_out, obs_out, st);
}

extern "C" int nmmo_sample_actions(nmmo_handle *h, uint64_t seed, int32_t *actions_dev, void *stream) {
  if (!h || !actions_dev) return fail(NM_ERR_ARG, "null argument");
  CU(cudaSetDevice(h->device));
  NmParams prm = h->prm;
  int threads = 256, NW = threads / 32;
  long long n_agents = (long long)prm.E * prm.P;
  int blocks = (int)std::min<long long>((n_agents + NW - 1) / NW, 148LL * 8 * 4);
  size_t smem = (size_t)NW * a16(prm.L.m_end);
  nmmo_sample_kernel<<<blocks, threads, smem, (cudaStream_t)stream>>>(prm, seed, actions_dev);
  CU(cudaGetLastError());
  return NM_OK;
}

extern "C" int nmmo_forage_actions(nmmo_handle *h, uint64_t seed, int32_t *actions_dev, void *stream) {
  if (!h || !actions_dev) return fail(NM_ERR_ARG, "null argument");
  if ((uintptr_t)actions_dev & 15) return fail(NM_ERR_ARG, "actions must be 16-byte aligned");
  CU(cudaSetDevice(h->device));
  NmParams prm = h->prm;
  const int threads = 256, NW = threads / 32;
  const long long n_agents = (long long)prm.E * prm.P;
  const int blocks = (int)std::min<long long>((n_agents + NW - 1) / NW, 148LL * 8 * 4);
  nmmo_forage_kernel<<<blocks, threads, 0, (cudaStream_t)stream>>>(prm, seed, actions_dev);
  CU(cudaGetLastError());
  return NM_OK;
}

extern "C" void *nmmo_obs_ptr(nmmo_handle *h) { return h->prm.obs; }
extern "C" void *nmmo_reward_ptr(nmmo_handle *h) { return h->prm.rew; }
extern "C" void *nmmo_terminated_ptr(nmmo_handle *h) { return h->prm.term; }
extern "C" void *nmmo_truncated_ptr(nmmo_handle *h) { return h->prm.trunc; }
extern "C" void *nmmo_mask_ptr(nmmo_handle *h) { return h->prm.mask; }
extern "C" void *nmmo_info_ptr(nmmo_handle *h) { return h->prm.info; }
extern "C" void *nmmo_info_valid_ptr(nmmo_handle *h) { return h->prm.info_valid; }
extern "C" void *nmmo_episode_done_ptr(nmmo_handle *h) { return h->prm.episode_done; }
extern "C" void *nmmo_task_id_ptr(nmmo_handle *h) { return h->prm.task_id; }
extern "C" void *nmmo_task_embed_ptr(nmmo_handle *h) { return (void *)h->prm.embed; }
extern "C" const char *nmmo_step_kernel_name(nmmo_handle *h) { return step_kernel(h, h->prm).name; }
extern "C" const char *nmmo_obs_kernel_name(nmmo_handle *h) { return obs_kernel(h, h->prm).name; }
extern "C" int nmmo_obs_stride(nmmo_handle *h) { return h->prm.L.stride; }
extern "C" int nmmo_num_envs(nmmo_handle *h) { return h->prm.E; }
extern "C" int nmmo_num_agents(nmmo_handle *h) { return h->prm.P; }

extern "C" int nmmo_inject_rng(nmmo_handle *h, int env, const uint64_t *keys, const uint32_t *vals, int n) {
  if (!h || env < 0 || env >= h->prm.E || n < 0 || (n > 0 && (!keys || !vals))) return fail(NM_ERR_ARG, "bad argument");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  auto &v = h->inj[env];
  v.clear();
  for (int i = 0; i < n; i++) v.emplace_back(keys[i], vals[i]);
  std::sort(v.begin(), v.end());
  std::vector<uint64_t> K; std::vector<uint32_t> V; std::vector<int32_t> off(h->prm.E + 1, 0);
  for (int e = 0; e < h->prm.E; e++) {
    off[e] = (int32_t)K.size();
    for (auto &kv : h->inj[e]) { K.push_back(kv.first); V.push_back(kv.second); }
  }
  off[h->prm.E] = (int32_t)K.size();
  if (h->d_inj_keys) { cudaFree(h->d_inj_keys); h->d_inj_keys = nullptr; }
  if (h->d_inj_vals) { cudaFree(h->d_inj_vals); h->d_inj_vals = nullptr; }
  if (K.empty()) { h->prm.inj_off = nullptr; h->prm.inj_keys = nullptr; h->prm.inj_vals = nullptr; return NM_OK; }
  CU(cudaMalloc((void **)&h->d_inj_keys, K.size() * sizeof(uint64_t)));
  CU(cudaMalloc((void **)&h->d_inj_vals, V.size() * sizeof(uint32_t)));
  CU(cudaMemcpy(h->d_inj_keys, K.data(), K.size() * sizeof(uint64_t), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_inj_vals, V.data(), V.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
  CU(cudaMemcpy(h->d_inj_off, off.data(), off.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
  h->prm.inj_off = h->d_inj_off; h->prm.inj_keys = h->d_inj_keys; h->prm.inj_vals = h->d_inj_vals;
  return NM_OK;
}

extern "C" int nmmo_snapshot(nmmo_handle *h, int env, int16_t *ent, int16_t *items, uint8_t *map, int32_t *scalars16) {
  if (!h || env < 0 || env >= h->prm.E) return fail(NM_ERR_ARG, "bad argument");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  const NmParams &p = h->prm;
  if (ent) {
    const size_t ent_i16 = p.big ? (size_t)NM_BIG_ENT_STRIDE * p.R : (size_t)EA_N * p.R;
    std::vector<int16_t> soa(ent_i16);
    CU(cudaMemcpy(soa.data(), p.ent + (size_t)env * ent_i16, soa.size() * 2, cudaMemcpyDeviceToHost));
    auto at = [&](int k, int r) -> int16_t { return p.big ? soa[(size_t)VBig::ent_idx(k, r, p.R)] : soa[(size_t)VSmall::ent_idx(k, r, p.R)]; };
    for (int r = 0; r < p.R; r++) {
      bool empty = at(EA_STATUS, r) == ES_EMPTY;
      for (int k = 0; k < EA_N; k++) ent[(size_t)r * EA_N + k] = empty ? 0 : at(k, r);
    }
  }
  if (items) {
    std::vector<int16_t> soa((size_t)IS_N * p.CAP);
    CU(cudaMemcpy(soa.data(), p.item + (size_t)env * IS_N * p.CAP, soa.size() * 2, cudaMemcpyDeviceToHost));
    for (int i = 0; i < p.CAP; i++)
      for (int k = 0; k < IS_N; k++) items[(size_t)i * IS_N + k] = soa[(size_t)k * p.CAP + i];
    int32_t hi = 0;      // rows >= SC_ITEM_HI are free: their bytes in HBM are stale, report them empty
    CU(cudaMemcpy(&hi, p.scalars + (size_t)env * NM_SC_N + SC_ITEM_HI, sizeof(hi), cudaMemcpyDeviceToHost));
    for (int i = std::max(hi, 0); i < p.CAP; i++)
      for (int k = 0; k < IS_N; k++) items[(size_t)i * IS_N + k] = 0;
  }
  if (map) {      // the live map is packed 4 bits per tile; the caller gets one byte per tile
    size_t nt = (size_t)p.S * p.S;
    std::vector<uint8_t> packed(nt / 2);
    CU(cudaMemcpy(packed.data(), p.map + (size_t)env * (nt / 2), nt / 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < nt; i++) map[i] = (packed[i >> 1] >> ((i & 1) * 4)) & 15;
  }
  if (scalars16) CU(cudaMemcpy(scalars16, p.scalars + (size_t)env * NM_SC_N, sizeof(int32_t) * NM_SC_N, cudaMemcpyDeviceToHost));
  return NM_OK;
}

extern "C" int nmmo_task_state(nmmo_handle *h, int env, int32_t *task_id, int32_t *completed, int32_t *reward_signals,
                               double *max_progress) {
  if (!h || env < 0 || env >= h->prm.E) return fail(NM_ERR_ARG, "bad argument");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  const NmParams &p = h->prm;
  const size_t P = p.P;
  std::vector<int32_t> st(P * ST_N);
  std::vector<double> ds(P * DS_N);
  CU(cudaMemcpy(st.data(), p.stats + (size_t)env * P * ST_N, st.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
  CU(cudaMemcpy(ds.data(), p.dstats + (size_t)env * P * DS_N, ds.size() * sizeof(double), cudaMemcpyDeviceToHost));
  if (task_id) CU(cudaMemcpy(task_id, p.task_id + (size_t)env * P, P * sizeof(int32_t), cudaMemcpyDeviceToHost));
  for (size_t a = 0; a < P; a++) {
    if (completed) completed[a] = st[a * ST_N + ST_TASK_DONE];
    if (reward_signals) reward_signals[a] = st[a * ST_N + ST_REWARD_SIGNALS];
    if (max_progress) max_progress[a] = ds[a * DS_N + DS_MAX_PROGRESS];
  }
  return NM_OK;
}

extern "C" int nmmo_stats(nmmo_handle *h, double *sums, double *counts, uint64_t *counters, int clear) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  std::vector<double> rep((size_t)NM_AGG_REP * 2 * IN_N);
  CU(cudaMemcpy(rep.data(), h->prm.agg, rep.size() * sizeof(double), cudaMemcpyDeviceToHost));
  double agg[2 * IN_N] = {0};
  for (int r = 0; r < NM_AGG_REP; r++)
    for (int i = 0; i < 2 * IN_N; i++) agg[i] += rep[(size_t)r * 2 * IN_N + i];
  // slot IN_N + 0 counts finished agents; only the max-level keys can be absent (NaN) and keep their own count
  for (int i = 1; i < IN_N; i++)
    if (!(i >= IN_MAXLVL_ARMOR && i <= IN_MAXLVL_CONSUMABLE)) agg[IN_N + i] = agg[IN_N];
  if (sums) memcpy(sums, agg, sizeof(double) * IN_N);
  if (counts) memcpy(counts, agg + IN_N, sizeof(double) * IN_N);
  if (counters) CU(cudaMemcpy(counters, h->prm.counters, sizeof(uint64_t) * 8, cudaMemcpyDeviceToHost));
  if (clear) { CU(cudaMemset(h->prm.agg, 0, rep.size() * sizeof(double))); CU(cudaMemset(h->prm.counters, 0, sizeof(uint64_t) * 8)); }
  return NM_OK;
}

// per-kernel timing: enable, run steps, then read the mean durations of the two kernels
extern "C" int nmmo_timing(nmmo_handle *h, int enable) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  h->timing = enable != 0;
  h->ev_used = 0;
  return NM_OK;
}
extern "C" int nmmo_timing_read(nmmo_handle *h, double *step_ms, double *obs_ms, int *n_launches) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  double a = 0, b = 0;
  int n = (int)(h->ev_used / 3);
  for (int i = 0; i < n; i++) {
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, h->ev[3 * i], h->ev[3 * i + 1])); a += ms;
    CU(cudaEventElapsedTime(&ms, h->ev[3 * i + 1], h->ev[3 * i + 2])); b += ms;
  }
  if (step_ms) *step_ms = n ? a / n : 0;
  if (obs_ms) *obs_ms = n ? b / n : 0;
  if (n_launches) *n_launches = n;
  h->ev_used = 0;
  return NM_OK;
}

// per-phase clock profile of the step kernel (development aid): enable allocates/clears the
// accumulators, read copies 64 counters (0..31 step kernel, 32..63 observation kernel) (SM clock cycles summed over CTAs) to the host
extern "C" int nmmo_profile(nmmo_handle *h, int enable, unsigned long long *out32) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());
  if (out32 && h->prm.prof) CU(cudaMemcpy(out32, h->prm.prof, 64 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  if (enable) {
    if (!h->prm.prof) { int rc = dalloc(h, &h->prm.prof, 64); if (rc) return rc; }
    CU(cudaMemset(h->prm.prof, 0, 64 * sizeof(unsigned long long)));
  } else h->prm.prof = nullptr;
  return NM_OK;
}

// 1 = the observation kernel rewrites every byte of every record each tick (dense mode, the
// HBM-roofline configuration); 0 (default) = only bytes that can differ from the record in HBM
extern "C" int nmmo_set_obs_full(nmmo_handle *h, int full) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  h->prm.obs_full = full != 0;
  return NM_OK;
}

// Built-in random policy: when `actions_dev_out` is non-NULL every observation pass also writes
// uniform-random valid actions (same draws as nmmo_sample_actions with this seed) into it, so a
// rollout with the random policy needs no sampler launch.  NULL switches it off.
extern "C" int nmmo_set_autosample(nmmo_handle *h, uint64_t seed, int32_t *actions_dev_out) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  h->prm.sample_out = actions_dev_out;
  h->prm.sample_seed = seed;
  return NM_OK;
}

// ------------------------------------------------------------------------------------------ environment state ----
extern "C" int nmmo_state_bytes(nmmo_handle *h, size_t *bytes) {
  if (!h || !bytes) return fail(NM_ERR_ARG, "null argument");
  *bytes = h->state.state_bytes;
  return NM_OK;
}

static int state_check_ids(nmmo_handle *h, const int32_t *env_ids, int n, const void *states, bool unique) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  if (n < 1) return fail(NM_ERR_ARG, "n must be at least 1");
  if (!env_ids || !states) return fail(NM_ERR_ARG, "null argument");
  std::vector<uint8_t> seen(unique ? h->prm.E : 0, 0);
  for (int i = 0; i < n; i++) {
    const int e = env_ids[i];
    if (e < 0 || e >= h->prm.E) return fail(NM_ERR_ARG, "env id " + std::to_string(e) + " out of range [0, " + std::to_string(h->prm.E) + ")");
    if (unique && seen[e]++) return fail(NM_ERR_ARG, "env id " + std::to_string(e) + " appears twice in a load");
  }
  if ((uintptr_t)states & 15) return fail(NM_ERR_ARG, "states must be 16-byte aligned");
  return NM_OK;
}

// save / load kernels over env_ids, NM_STATE_IDS envs per launch; blob j of the call is states + j * state_bytes
static int launch_state(nmmo_handle *h, bool save, const int32_t *env_ids, int n, uint8_t *states, cudaStream_t st) {
  NmStateArgs a = h->state;
  for (int k = 0; k < n; k += NM_STATE_IDS) {
    a.n = std::min(NM_STATE_IDS, n - k);
    memcpy(a.ids, env_ids + k, sizeof(int32_t) * a.n);
    const unsigned grid = (unsigned)a.n * a.n_chunks;
    uint8_t *blobs = states + (size_t)k * a.state_bytes;
    a.ev_n = h->prm.ev_n;
    if (save) nmmo_state_save_kernel<<<grid, NM_STATE_THREADS, 0, st>>>(a, blobs);
    else nmmo_state_load_kernel<<<grid, NM_STATE_THREADS, 0, st>>>(a, blobs);
    CU(cudaGetLastError());
  }
  return NM_OK;
}

extern "C" int nmmo_save_envs(nmmo_handle *h, const int32_t *env_ids, int n, uint8_t *states_dev, void *stream) {
  int rc = state_check_ids(h, env_ids, n, states_dev, false);
  if (rc) return rc;
  CU(cudaSetDevice(h->device));
  return launch_state(h, true, env_ids, n, states_dev, (cudaStream_t)stream);
}

extern "C" int nmmo_load_envs(nmmo_handle *h, const int32_t *env_ids, int n, const uint8_t *states_dev, void *stream) {
  int rc = state_check_ids(h, env_ids, n, states_dev, true);
  if (rc) return rc;
  if (h->timing || h->prm.prof)
    return fail(NM_ERR_STATE, "per-kernel timing and the phase profiler describe whole-handle launches: switch them off to load envs");
  CU(cudaSetDevice(h->device));
  const cudaStream_t st = (cudaStream_t)stream;
  const NmStateArgs &a = h->state;
  // every header is checked before any device state is touched: an NM_ERR_ARG return leaves the handle as it was
  CU(cudaStreamSynchronize(st));
  std::vector<NmStateHeader> hd(n);
  CU(cudaMemcpy2DAsync(hd.data(), sizeof(NmStateHeader), states_dev, a.state_bytes, sizeof(NmStateHeader), n,
                       cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  static const char *fam[2] = {"small", "big"};
  for (int i = 0; i < n; i++) {
    const NmStateHeader &x = hd[i];
    const std::string which = "state " + std::to_string(i) + ": ";
    if (x.magic != NM_STATE_MAGIC) return fail(NM_ERR_ARG, which + "not an environment state blob (bad magic)");
    if (x.version != NM_STATE_VERSION)
      return fail(NM_ERR_ARG, which + "format version " + std::to_string(x.version) + "; this build reads version " + std::to_string(NM_STATE_VERSION));
    if (x.family != a.hdr.family)
      return fail(NM_ERR_ARG, which + "saved by a " + std::string(x.family <= 1 ? fam[x.family] : "unknown") + "-family handle; this handle runs the " +
                              fam[a.hdr.family] + " family");
    if (x.state_bytes != a.state_bytes)
      return fail(NM_ERR_ARG, which + "a blob of " + std::to_string(x.state_bytes) + " bytes; this handle's are " + std::to_string(a.state_bytes));
    if (x.digest != a.hdr.digest)
      return fail(NM_ERR_ARG, which + "digest mismatch: saved by a handle created with another config, maps, task table or task embeddings");
  }
  rc = launch_state(h, false, env_ids, n, (uint8_t *)states_dev, st);
  if (rc) return rc;
  // the loaded envs' records, ActionTargets masks and built-in-policy rows, rebuilt by the observation kernel as after a
  // reset; the other envs of the span get the bytes they already hold
  const int lo = *std::min_element(env_ids, env_ids + n), hi = *std::max_element(env_ids, env_ids + n) + 1;
  NmParams prm = h->prm;
  return launch_obs_kernel(h, prm, st, lo, hi);
}

// ------------------------------------------------------------------------------------------------ event log ----
extern "C" int nmmo_set_event_log(nmmo_handle *h, int enable) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());      // no step in flight may write the staging while it changes
  NmParams &p = h->prm;
  if (!enable) {
    if (p.ev_log) { CU(cudaFree(p.ev_log)); CU(cudaFree(p.ev_n)); CU(cudaFree(h->ev_off)); }
    p.ev_log = nullptr; p.ev_n = nullptr; h->ev_off = nullptr;
    return NM_OK;
  }
  if (!p.ev_log) {
    uint2 *log = nullptr; int32_t *n = nullptr, *off = nullptr;
    cudaError_t e = cudaMalloc((void **)&log, (size_t)p.E * p.ev_cap * sizeof(uint2));
    if (e == cudaSuccess) e = cudaMalloc((void **)&n, (size_t)p.E * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc((void **)&off, (size_t)p.E * sizeof(int32_t));
    if (e != cudaSuccess) {
      cudaFree(log); cudaFree(n); cudaFree(off);
      return fail(NM_ERR_CUDA, std::string("event log staging: ") + cudaGetErrorString(e));
    }
    p.ev_log = log; p.ev_n = n; h->ev_off = off;
  }
  CU(cudaMemset(p.ev_n, 0, (size_t)p.E * sizeof(int32_t)));
  return NM_OK;
}

extern "C" int nmmo_events(nmmo_handle *h, int env_lo, int env_hi, int32_t *rows_dev, int cap, int32_t *count_dev, void *stream) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  const NmParams &p = h->prm;
  if (!p.ev_log) return fail(NM_ERR_STATE, "the event log is off: nmmo_set_event_log(h, 1) first");
  if (env_lo < 0 || env_hi > p.E || env_lo >= env_hi) return fail(NM_ERR_ARG, "env range must satisfy 0 <= env_lo < env_hi <= E");
  if (cap < 0) return fail(NM_ERR_ARG, "cap must be >= 0");
  if (!count_dev || (cap > 0 && !rows_dev)) return fail(NM_ERR_ARG, "null argument");
  if (((uintptr_t)rows_dev | (uintptr_t)count_dev) & 3) return fail(NM_ERR_ARG, "rows and count must be 4-byte aligned");
  CU(cudaSetDevice(h->device));
  const cudaStream_t st = (cudaStream_t)stream;
  nmmo_events_scan_kernel<<<1, NM_EV_SCAN_THREADS, 0, st>>>(p.ev_n, env_lo, env_hi, h->ev_off, count_dev);
  CU(cudaGetLastError());
  if (cap == 0) return NM_OK;
  NmEventsArgs a;
  a.ev_log = p.ev_log; a.ev_n = p.ev_n; a.off = h->ev_off; a.scalars = p.scalars;
  a.ev_cap = p.ev_cap; a.P = p.P; a.lo = env_lo; a.rows = rows_dev; a.cap = cap;
  nmmo_events_kernel<<<env_hi - env_lo, NM_EV_THREADS, (size_t)(p.P + p.ev_cap) * sizeof(int), st>>>(a);
  CU(cudaGetLastError());
  return NM_OK;
}

// ------------------------------------------------------------------------------------ next-episode values ----
extern "C" int nmmo_set_next_episodes(nmmo_handle *h, int enable) {
  if (!h) return fail(NM_ERR_ARG, "null handle");
  CU(cudaSetDevice(h->device));
  CU(cudaDeviceSynchronize());      // no step in flight may read or clear the flags while they change
  NmParams &p = h->prm;
  if (!enable) {
    if (p.next_flags) { CU(cudaFree(p.next_flags)); CU(cudaFree(p.next_seed)); CU(cudaFree(p.next_map)); CU(cudaFree(p.next_task)); }
    p.next_flags = nullptr; p.next_seed = nullptr; p.next_map = nullptr; p.next_task = nullptr;
    return NM_OK;
  }
  const size_t E = p.E, P = p.P;
  if (!p.next_flags) {
    uint8_t *f = nullptr; uint64_t *sd = nullptr; int32_t *m = nullptr, *t = nullptr;
    cudaError_t e = cudaMalloc((void **)&f, E);
    if (e == cudaSuccess) e = cudaMalloc((void **)&sd, E * sizeof(uint64_t));
    if (e == cudaSuccess) e = cudaMalloc((void **)&m, E * sizeof(int32_t));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t, E * P * sizeof(int32_t));
    if (e != cudaSuccess) {
      cudaFree(f); cudaFree(sd); cudaFree(m); cudaFree(t);
      return fail(NM_ERR_CUDA, std::string("next-episode buffers: ") + cudaGetErrorString(e));
    }
    p.next_flags = f; p.next_seed = sd; p.next_map = m; p.next_task = t;
    CU(cudaMemset(p.next_seed, 0, E * sizeof(uint64_t)));
    CU(cudaMemset(p.next_map, 0, E * sizeof(int32_t)));
    CU(cudaMemset(p.next_task, 0, E * P * sizeof(int32_t)));
  }
  CU(cudaMemset(p.next_flags, 0, E));
  CU(cudaDeviceSynchronize());
  return NM_OK;
}
extern "C" void *nmmo_next_flags_ptr(nmmo_handle *h) { return h->prm.next_flags; }
extern "C" void *nmmo_next_seed_ptr(nmmo_handle *h) { return h->prm.next_seed; }
extern "C" void *nmmo_next_map_ptr(nmmo_handle *h) { return h->prm.next_map; }
extern "C" void *nmmo_next_task_ptr(nmmo_handle *h) { return h->prm.next_task; }
