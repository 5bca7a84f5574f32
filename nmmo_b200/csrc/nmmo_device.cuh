// nmmo_device.cuh -- device-side state description and small helpers shared by the kernels.
//
// Layout in HBM (one handle = E lock-stepped environments on one GPU), all per-env blocks
// contiguous and 16-byte aligned so a CTA pulls its environment into shared memory with
// three cp.async.bulk (TMA 1-D) copies and pushes it back the same way:
//   ent   int16 [E][EA_N][R]      structure-of-arrays entity table (players rows 0..P-1, NPCs after)
//   item  int16 [E][IS_N][CAP]    item table (only stored columns; stats derive from type+level);
//                                 rows >= scalars[SC_ITEM_HI] are free and their content is unspecified
//   map   uint8 [E][S*S/2]        current tile materials, 4 bits per tile (16 materials)
// plus small per-agent blocks (stats, unique-event bitsets, task state) and the output
// tensors (obs records, reward, terminated, truncated, mask, episode info).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/nmmo_spec.h"

#define NM_EV_CAP 1024          // per-env per-tick event ring (shared memory)
#define NM_STEP_THREADS 256
#ifndef NM_STEP4_THREADS
#define NM_STEP4_THREADS 192      // step kernel, four environments per CTA: threads per environment (768 per CTA, 80 registers)
#endif
#ifndef NM_OBS_THREADS
#define NM_OBS_THREADS 512         // observation kernels: 16 warps per CTA ...
#define NM_OBS_CTAS_PER_SM 2       // ... two CTAs per SM
#endif
#define NM_SC_N 16              // per-env int32 scalars
#define NM_DEPL_CAP 1024         // per-env list of depleted tiles kept across ticks (falls back to a map scan beyond)
#define NM_AGG_REP 256           // replicas of the finished-agent sums (contention spreading)
// big family (nmmo_step_big_kernel / nmmo_obs_big_kernel: up to 1024 players, 3072 entities, 1023^2 tiles per env)
#define NM_BIG_THREADS 1024
#define NM_BIG_EV_CAP 4096
#define NM_BIG_DEPL_CAP 4096
#define NM_BIG_ENT_STRIDE 48     // int16 per row of the row-major entity table (EA_N = 44, padded to 96 bytes)
#define NM_BIG_OBS_AGENTS 128    // agents per CTA of the big observation kernel
#define NM_OBS_CELL 16           // observation kernel: side of the cells the alive rows are bucketed by (>= 2 * vision)
#ifndef NM_OBS_BATCH
#define NM_OBS_BATCH 8
#endif
//      NM_OBS_BATCH:           // observation kernel: agents per warp whose built-in-policy heads are resolved together (5 x 12 heads = 60 lanes)
#ifndef NM_OBS_DEAL_NUM
#define NM_OBS_DEAL_NUM 8           // observation kernel: eighths of the work list dealt round-robin, the rest pulled (measured: 4/8 0.532 ms, 6/8 0.530, 7/8 0.528, all dealt 0.528)
#endif
#ifndef NM_OBS_PREFETCH_AHEAD
#define NM_OBS_PREFETCH_AHEAD 64
#endif
//      NM_OBS_PREFETCH_AHEAD:  // observation kernel (small family): a CTA prefetches into L2 the tables of the env this many CTAs later
#ifndef NM_OBS_EROWS
#define NM_OBS_EROWS 8             // observation kernel (small family): Entity rows a warp stages per group (8 or 16)
#endif
#ifndef NM_OBS_ENT_SKEW
#define NM_OBS_ENT_SKEW 8
#endif
//      NM_OBS_ENT_SKEW:         // observation kernel (small family): int16 of padding between staged entity columns
#define OM_NONZERO (1u << 16)
#define OM_TASK (1u << 17)

enum nm_scalar { SC_TICK = 0, SC_DONE, SC_NEXT_NPC_ID, SC_N_DANGER, SC_MAP_ID, SC_EPISODE, SC_FRESH,
                 SC_ERROR, SC_NEED_RESET, SC_EXPLICIT_MAP, SC_EXPLICIT_TASKS,
                 SC_ITEM_HI /* rows >= this are free; multiple of 8 */,
                 SC_N_DEPL /* entries of the depleted-tile list; -1 = unknown, rebuild it from a map scan */ };

struct NmParams {
  // the config vector, rounded up to whole 16-byte words: the members after it keep their offsets modulo 16 whatever
  // NC_COUNT is, and with them the kernels' merged parameter loads (e.g. two reward weights per 128-bit constant load)
  int32_t cfg[(NC_COUNT + 3) & ~3];
  double fcfg[NF_COUNT];
  nm_obs_layout L;
  int E, P, N, R, S, CAP, n_maps, n_tasks;
  int ICAP;                    // item rows staged in shared memory (the tail is used in HBM)
  // state
  int16_t *ent, *item;
  uint8_t *map;
  const uint8_t *maps;
  int32_t *scalars;            // [E][NM_SC_N]
  uint64_t *seed;              // [E]
  int16_t *danger;             // [E][N]
  void *depl;                  // [E][depleted-list capacity] tile indices of the depleted tiles (unordered; uint16 small / uint32 big)
  uint8_t *ws; size_t ws_bytes;// big family: per-env workspace for the step kernel's rarely touched arrays
  int ev_cap;                  // events an env may emit per tick before the ring overflows (the family's ring size)
  int big;                     // 1 = big family (row-major entity table, tables used in place)
  int32_t *stats;              // [E][P][ST_N]
  double *dstats;              // [E][P][DS_N]
  uint32_t *uniq;              // [E][P][NM_UNIQ_WORDS]
  int32_t *task_id;            // [E][P]
  const int32_t *tasks;        // [T][NM_TASK_COLS]
  const uint16_t *embed;       // [T][task_dim]
  // rng injection
  const uint64_t *inj_keys; const uint32_t *inj_vals; const int32_t *inj_off;   // off [E+1]
  // io
  const int32_t *actions;      // [E][P][12]
  uint8_t *obs;                // [E*P][stride]
  float *rew; uint8_t *term, *trunc, *mask; float *info; uint8_t *info_valid; uint8_t *episode_done;
  double *agg;                 // [NM_AGG_REP][2][IN_N] sums and counts of finished-agent info
  unsigned long long *counters;// [8] slot-steps, alive-agent-steps, episodes, errors, obs-kernel bytes
  uint32_t *obs_meta;          // [E*P] what each obs record currently holds (incremental writer)
  int obs_full;                // 1 = rewrite every byte of every record each tick
  int32_t *sample_out;         // optional: the obs kernel also writes uniform-random valid actions here
  uint64_t sample_seed;
  unsigned long long *prof;    // optional [32] per-phase clock accumulators (NULL = off)
  int half_smem;               // step kernel: dynamic shared memory of one environment
  int no_depl_list;            // test hook: never trust the depleted-tile list (always rebuild it from a map scan)
  int envs_per_cta;            // step kernel: environments per CTA (4, 3, 2 or 1: as many as fit in shared memory)
  int mode;                    // 0 step (auto-reset finished envs), 1 reset flagged envs only
  int env_lo, env_hi;          // step and observation kernels: the environments this launch covers
  int act_env_lo;              // env whose actions are row 0 of `actions` (0 = a whole-handle buffer; nmmo_step_envs: its env_lo)
  int env_base;                // global env index of env 0 (multi-GPU sharding; seeds derive from it)
  // event log (nmmo_set_event_log; NULL = off): the step kernel keeps each env's events of the call here, the ring as
  // emitted, and their count (0 for an env the call resets); nmmo_events turns them into rows (nmmo_events.cu)
  uint2 *ev_log;               // [E][ev_cap]
  int32_t *ev_n;               // [E]
  // pending next-episode values (nmmo_set_next_episodes; NULL = off): an env's automatic reset takes the fields whose
  // nm_next bit is set in its flags byte from here, then clears the byte
  uint8_t *next_flags;         // [E]
  uint64_t *next_seed;         // [E]
  int32_t *next_map;           // [E]
  int32_t *next_task;          // [E][P] task-table rows (agent p reads its team leader's entry)
};

// The reference's default shape (config 2: 128 players, 256 NPCs, 160^2 map, N_ent 100, N_mkt 384, 12 inventory rows,
// 99 prices, 2048-d task, vision 7) as compile-time constants: with it every record offset, stride and divisor of the
// kernels folds into immediates.  nmmo_create selects the *_std kernels when the handle has this shape.
__host__ __device__ constexpr nm_obs_layout nm_std_layout() {
  nm_obs_layout L{};
  L.n_ent = 100; L.n_mkt = 384; L.n_inv = 12; L.n_price = 99; L.task_dim = 2048; L.win = 15;
  int o = 0;
  L.m_style = o; o += 3;
  L.m_target = o; o += L.n_ent + 1;
  L.m_buy = o; o += L.n_mkt + 1;
  L.m_destroy = o; o += L.n_inv + 1;
  L.m_give_item = o; o += L.n_inv + 1;
  L.m_give_target = o; o += L.n_ent + 1;
  L.m_gold_price = o; o += L.n_price;
  L.m_gold_target = o; o += L.n_ent + 1;
  L.m_move = o; o += NM_DIR_N;
  L.m_sell_item = o; o += L.n_inv + 1;
  L.m_sell_price = o; o += L.n_price;
  L.m_use = o; o += L.n_inv + 1;
  L.m_end = o;
  L.alg_bytes = o;
  o = (o + 15) & ~15;
  L.o_ids = o; o += 4; L.alg_bytes += 4; o = (o + 15) & ~15;
  L.o_entity = o; o += L.n_ent * EA_N_OBS * 2; L.alg_bytes += L.n_ent * EA_N_OBS * 2; o = (o + 15) & ~15;
  L.o_inventory = o; o += L.n_inv * IA_N_OBS * 2; L.alg_bytes += L.n_inv * IA_N_OBS * 2; o = (o + 15) & ~15;
  L.o_market = o; o += L.n_mkt * IA_N_OBS * 2; L.alg_bytes += L.n_mkt * IA_N_OBS * 2; o = (o + 15) & ~15;
  L.o_task = o; o += L.task_dim * 2; L.alg_bytes += L.task_dim * 2; o = (o + 15) & ~15;
  L.o_tile = o; o += L.win * L.win * 3 * 2; L.alg_bytes += L.win * L.win * 3 * 2;
  L.stride = (o + 127) & ~127;
  return L;
}
struct StdShape { static constexpr int P = 128, N = 256, R = 384, S = 160, CAP = 1536, ICAP = 256, NINV = 12, VIS = 7; };
// ... and the shape of BASELINE.json configs[4] (1024 players, 2048 NPCs, 544^2 map; same record layout) for the big family
struct StdShape5 { static constexpr int P = 1024, N = 2048, R = 3072, S = 544, CAP = 12288, ICAP = 0, NINV = 12, VIS = 7; };


// Engine defaults of nmmo.core.config [UPSTREAM] that the reference's Config never overrides (environment.py:14-49 sets
// PLAYER_N, NPC_N, HORIZON, MAP_*, TASK_EMBED_DIM, RESILIENT_POPULATION, SPAWN_IMMUNITY and the wrapper arguments only),
// as compile-time constants for the *_std kernel instantiations.  nm_cfg_std_value(i) < 0x7fffffff for every folded
// index; nmmo_create selects a *_std kernel only when the handle's vector equals this table at every folded index
// (tests/test_host.py checks the table against nmmo_b200/config.py make_config()).
#define NM_CFG_RUNTIME 0x7fffffff
__host__ __device__ constexpr int nm_cfg_std_value(int i) {
  switch (i) {
    case NC_MAP_BORDER: return 16;
    case NC_N_ENT_OBS: return 100;
    case NC_N_MKT_OBS: return 384;
    case NC_N_INV: return 12;
    case NC_N_PRICE: return 99;
    case NC_VISION: return 7;
    case NC_TASK_DIM: return 2048;
    case NC_NPC_VISION: return 5;
    case NC_RES_BASE: return 100;
    case NC_RES_DEPLETION: return 5;
    case NC_RES_STARVATION: return 10;
    case NC_RES_DEHYDRATION: return 10;
    case NC_RES_REGEN_THRESH: return 50;
    case NC_RES_HEALTH_RESTORE: return 10;
    case NC_RES_HARVEST_RESTORE: return 100;
    case NC_REACH: return 3;
    case NC_FREEZE_TIME: return 3;
    case NC_WEAK_NUM: return 3;
    case NC_WEAK_DEN: return 2;
    case NC_MINDMG_NUM: return 1;
    case NC_MINDMG_DEN: return 4;
    case NC_LEVEL_MAX: return 10;
    case NC_XP_COMBAT: return 6;
    case NC_XP_AMMO: return 15;
    case NC_XP_CONSUMABLE: return 30;
    case NC_BASE_DAMAGE: return 10;
    case NC_LEVEL_DAMAGE: return 5;
    case NC_BASE_DEFENSE: return 0;
    case NC_LEVEL_DEFENSE: return 5;
    case NC_EXP_THRESH0: return 0;
    case NC_EXP_THRESH0 + 1: return 30;
    case NC_EXP_THRESH0 + 2: return 72;
    case NC_EXP_THRESH0 + 3: return 124;
    case NC_EXP_THRESH0 + 4: return 184;
    case NC_EXP_THRESH0 + 5: return 251;
    case NC_EXP_THRESH0 + 6: return 324;
    case NC_EXP_THRESH0 + 7: return 403;
    case NC_EXP_THRESH0 + 8: return 488;
    case NC_EXP_THRESH0 + 9: return 578;
    case NC_NPC_SPAWN_ATTEMPTS: return 25;
    case NC_NPC_AGGR_PCT: return 80;
    case NC_NPC_NEUT_PCT: return 50;
    case NC_NPC_PASS_PCT: return 0;
    case NC_NPC_LEVEL_MIN: return 1;
    case NC_NPC_LEVEL_MAX: return 10;
    case NC_NPC_BASE_DEFENSE: return 0;
    case NC_NPC_LEVEL_DEFENSE: return 15;
    case NC_NPC_BASE_DAMAGE: return 15;
    case NC_NPC_LEVEL_DAMAGE: return 15;
    case NC_WEAPON_DROP_THR: return 107374182;
    case NC_WEAPON_BASE: return 5;
    case NC_WEAPON_LEVEL: return 5;
    case NC_AMMO_BASE: return 5;
    case NC_AMMO_LEVEL: return 10;
    case NC_TOOL_BASE: return 15;
    case NC_TOOL_LEVEL: return 0;
    case NC_ARMOR_BASE: return 0;
    case NC_ARMOR_LEVEL: return 3;
    case NC_RESTORE_BASE: return 50;
    case NC_RESTORE_LEVEL: return 5;
    case NC_RESPAWN_FOILAGE: return 107374182;
    case NC_RESPAWN_ORE: return 429496729;
    case NC_RESPAWN_TREE: return 450971566;
    case NC_RESPAWN_CRYSTAL: return 429496729;
    case NC_RESPAWN_HERB: return 85899345;
    case NC_RESPAWN_FISH: return 85899345;
    case NC_ALLOW_OCCUPIED: return 0;      // one entity per tile (DESIGN.md section 7); the reference's Config never sets it
    case NC_BASE_GOLD: return 1;
    case NC_LISTING_DURATION: return 3;
    // death fog: off (None) in every configuration the reference ships, so the *_std kernels compile it out; a handle with
    // fog on fails has_std_shape and runs the generic instantiation of the same source
    case NC_DEATH_FOG: return -1;
    case NC_DEATH_FOG_SPEED: return 1;
    case NC_DEATH_FOG_FINAL_SIZE: return 8;
    default: return NM_CFG_RUNTIME;      // shape entries (PLAYER_N, NPC_N, MAP_CENTER, MAP_SIZE, ITEM_CAP), HORIZON, RESILIENT_N,
                                         // SPAWN_IMMUNITY, the wrapper arguments and the workload knobs stay run-time
  }
}
// The config vector as the kernels see it: c[NC_X] with a literal index folds to the constant in a *_std instantiation
// (the accessor is inlined, the switch above disappears); c.p[...] is the plain vector for run-time indices.
template <bool STD>
struct NmCfg {
  const int32_t *p;
  __host__ __device__ __forceinline__ int operator[](int i) const {
#ifdef NM_NO_CFG_FOLD
    return p[i];
#else
    return (STD && nm_cfg_std_value(i) != NM_CFG_RUNTIME) ? nm_cfg_std_value(i) : p[i];
#endif
  }
};

// Observation kernel: whether the per-agent pre-pass runs for R table rows and AP agents per CTA -- at most 32 row-bitmap
// words per agent, and room for the AP agents' bitmaps in the built-in policy's batch words.  obs_body carves its
// per-agent lists where it does, and nmmo_create sizes the kernel's shared memory by it.
__host__ __device__ __forceinline__ bool nm_obs_pre_ok(int R, int AP) {
  const int RW = ((R + 31) & ~31) >> 5;
  return RW <= 32 && (size_t)AP * RW * 4 <= (size_t)(NM_OBS_THREADS >> 5) * NM_OBS_BATCH * 33 * 4;
}

// ------------------------------------------------------------------------- rng ------
__host__ __device__ __forceinline__ uint64_t nm_mix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ULL;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ uint64_t nm_hash64(uint64_t seed, uint32_t tick, uint32_t site,
                                                      uint32_t idx, uint32_t k) {
  uint64_t key = nm_rng_key(tick, site, idx, k);
  return nm_mix64(nm_mix64(seed ^ key) + key * 0xD6E8FEB86659FD93ULL);
}
__host__ __device__ __forceinline__ uint32_t nm_hash_draw(uint64_t seed, uint32_t tick, uint32_t site,
                                                         uint32_t idx, uint32_t k) {
  return (uint32_t)(nm_hash64(seed, tick, site, idx, k) >> 32);
}
// action sampler: one 64-bit hash per agent, murmur3 fmix32 per head
__host__ __device__ __forceinline__ uint32_t nm_action_draw(uint64_t base, int head) {
  uint32_t x = (uint32_t)base + (uint32_t)(base >> 32) * (uint32_t)(2 * head + 1);
  x ^= x >> 16; x *= 0x85EBCA6Bu; x ^= x >> 13; x *= 0xC2B2AE35u; x ^= x >> 16;
  return x;
}
__device__ __forceinline__ int nm_bounded(uint32_t u, int n) { return (int)(((uint64_t)u * (uint64_t)n) >> 32); }

// ----------------------------------------------------------------- async copies -----
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity) {
  uint32_t ok;
  asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
               : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// TMA 1-D bulk copy global -> shared, completion on an mbarrier (SASS: UBLKCP)
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// TMA 1-D bulk copy shared -> global
__device__ __forceinline__ void bulk_s2g(void *dst, const void *src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(smem_u32(src)), "r"(bytes) : "memory");
}
// TMA 1-D bulk prefetch global -> L2 (fire and forget)
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ------------------------------------------------------------------- materials ------
__device__ __forceinline__ int nm_impassible(int m) { return (NM_IMPASSIBLE_MASK >> m) & 1; }
__device__ __forceinline__ int nm_iabs(int x) { return x < 0 ? -x : x; }
__device__ __forceinline__ int nm_linf(int r0, int c0, int r1, int c1) { return max(nm_iabs(r0 - r1), nm_iabs(c0 - c1)); }

// ----------------------------------------------------------------------- items ------
__device__ __forceinline__ bool it_armor(int t) { return t >= IT_HAT && t <= IT_BOTTOM; }
__device__ __forceinline__ bool it_weapon(int t) { return t >= IT_SPEAR && t <= IT_WAND; }
__device__ __forceinline__ bool it_tool(int t) { return t >= IT_ROD && t <= IT_CHISEL; }
__device__ __forceinline__ bool it_ammo(int t) { return t >= IT_WHETSTONE && t <= IT_RUNES; }
__device__ __forceinline__ bool it_consumable(int t) { return t == IT_RATION || t == IT_POTION; }

// derived item columns (nmmo/systems/item.py constructors [UPSTREAM])
template <class C>
__device__ __forceinline__ int item_attack(const C &c, int type, int level, int style) {
  if (it_weapon(type) && type - IT_SPEAR == style) return c[NC_WEAPON_BASE] + level * c[NC_WEAPON_LEVEL];
  if (it_ammo(type) && type - IT_WHETSTONE == style) return c[NC_AMMO_BASE] + level * c[NC_AMMO_LEVEL];
  return 0;
}
template <class C>
__device__ __forceinline__ int item_defense(const C &c, int type, int level) {
  if (it_armor(type)) return c[NC_ARMOR_BASE] + level * c[NC_ARMOR_LEVEL];
  if (it_tool(type)) return c[NC_TOOL_BASE] + level * c[NC_TOOL_LEVEL];
  return 0;
}
// full 16-column observed item row
template <class C>
__device__ __forceinline__ void item_obs_row(const C &c, int row, int type, int level, int owner, int qty,
                                             int equipped, int price, int16_t out[IA_N_OBS]) {
#pragma unroll
  for (int k = 0; k < IA_N_OBS; k++) out[k] = 0;
  out[IA_ID] = (int16_t)(row + 1); out[IA_TYPE] = (int16_t)type; out[IA_OWNER] = (int16_t)owner;
  out[IA_LEVEL] = (int16_t)level; out[IA_QUANTITY] = (int16_t)qty; out[IA_EQUIPPED] = (int16_t)equipped;
  out[IA_LISTED_PRICE] = (int16_t)price;
  int d = item_defense(c, type, level);
  out[IA_MELEE_DEFENSE] = out[IA_RANGE_DEFENSE] = out[IA_MAGE_DEFENSE] = (int16_t)d;
  out[IA_MELEE_ATTACK] = (int16_t)item_attack(c, type, level, 0);
  out[IA_RANGE_ATTACK] = (int16_t)item_attack(c, type, level, 1);
  out[IA_MAGE_ATTACK] = (int16_t)item_attack(c, type, level, 2);
  int restore = c[NC_RESTORE_BASE] + level * c[NC_RESTORE_LEVEL];
  if (type == IT_RATION) out[IA_RESOURCE_RESTORE] = (int16_t)restore;
  if (type == IT_POTION) out[IA_HEALTH_RESTORE] = (int16_t)restore;
}

__device__ __forceinline__ int nm_dense_event(int code) {
  switch (code) {
    case EV_EAT_FOOD: return 0; case EV_DRINK_WATER: return 1; case EV_GO_FARTHEST: return 2;
    case EV_SCORE_HIT: return 3; case EV_PLAYER_KILL: return 4; case EV_CONSUME_ITEM: return 5;
    case EV_GIVE_ITEM: return 6; case EV_DESTROY_ITEM: return 7; case EV_HARVEST_ITEM: return 8;
    case EV_EQUIP_ITEM: return 9; case EV_LOOT_ITEM: return 10; case EV_GIVE_GOLD: return 11;
    case EV_LIST_ITEM: return 12; case EV_EARN_GOLD: return 13; case EV_BUY_ITEM: return 14;
    case EV_LOOT_GOLD: return 15; case EV_LEVEL_UP: return 16;
  }
  return -1;
}

static __constant__ int c_dir_dr[5] = {-1, 1, 0, 0, 0};   // North South East West Stay
static __constant__ int c_dir_dc[5] = {0, 0, 1, -1, 0};
