// nmmo_step.cu -- one thread group steps one environment: the whole Realm.step + reward/stat wrapper.
//
// Two instantiations of the same phases (struct VSmall / VBig below):
//   nmmo_step_kernel      256 threads per environment, two environments per CTA, every table in shared memory
//                         (PLAYER_N <= 256, P + N <= 512, map <= 255^2: BASELINE.json configs 1-4);
//                         nmmo_step3_kernel / nmmo_step4_kernel run three / four environments per CTA (VSmall3 / VSmall4);
//   nmmo_step_big_kernel  1024 threads per environment, one environment per CTA; the entity table (row-major), the
//                         item table and the tile map stay in HBM / L2 and only the hot indices (occupancy bitmap,
//                         position index, attack lists, inventories) live in shared memory
//                         (PLAYER_N <= 1024, P + N <= 3072, map <= 1023^2: configs[4], 1024 agents per env).
//
// What it replaces in the reference (all per-env, per-agent Python today):
//   nmmo.Env.step  (call site reinforcement_learning/stat_wrapper.py:64)   -> phases 0..13
//   BaseStatWrapper.step / _process_stats_and_early_stop (stat_wrapper.py:57-185),
//   process_event_log (:216-288), count_unique_events (:295-310)           -> phases 14..15
//   agent_zoo/{takeru,neurips23_start_kit,yaofeng}/reward_wrapper.py reward hooks  -> phase 15
//
// Execution model.  The environment's tables (entity table, 4-bit tile map, the live prefix of the
// item table) are pulled into shared memory by TMA bulk copies, every phase runs out of shared
// memory, and the tables are pushed back with bulk stores.  Phases whose reference semantics are
// order-free across agents (validation, NPC decide, resource update, Use, Destroy, Sell, cull,
// respawn, event folding, rewards) run one thread per entity.  Phases the reference executes in
// entity-id order keep that order exactly: harvest drops and Buy / Give by ballot-compacted
// sequential sections, Attack by rounds over entity-disjoint attacks, Move by a local decision per
// mover from a position index (see the comments at each phase).
//
// What the kernel's time follows (DESIGN.md 4.1): the code an environment walks per tick and the number of
// barrier-delimited segments on its critical path, not the bytes it moves.  Hence: short per-row loops are
// kept rolled (#pragma unroll 1; nvcc would unroll them four times for one or two trips), phases nobody asked
// for are skipped together with their barriers (`todo` mask), and row walks with ballots are spread over all
// warps with per-chunk counts and one barrier instead of being done by warp 0 alone.
#include "nmmo_device.cuh"

namespace {

// ---- the two kernel families -------------------------------------------------------------------------------------
struct VSmall {
  static constexpr int kThreads = NM_STEP_THREADS;      // per environment
  static constexpr int kRowsPerThread = 2;              // P + N <= 2 * kThreads
  static constexpr int kChunkIters = 1;                 // 32-row chunks per lane in the per-chunk prefix sums (<= 32 chunks)
  static constexpr int kEvCap = NM_EV_CAP, kDeplCap = NM_DEPL_CAP, kNpcHash = 512, kTblSlots = 1024;
  static constexpr bool kGlobalTables = false;          // tables are staged in shared memory by TMA bulk copies
  static constexpr bool kItemsInPlace = false;          // ... including the live prefix of the item table and the event ring
  static constexpr bool kScratchInWs = false;           // true: the per-tick arrays of VSmall4 below live in the HBM workspace
  static constexpr bool kStd = false;                   // true: a known shape (Shape) as compile-time constants
  typedef StdShape Shape;
  typedef uint16_t tile_t;                              // a tile index r * S + c
  // structure-of-arrays entity table: column-major inside the env (bank-conflict-free per-thread column access)
  static __host__ __device__ __forceinline__ int ent_idx(int col, int row, int R) { return col * R + row; }
};
// Small family, three environments per CTA: the item table and the event ring (30 KB of the 105 KB an environment
// needs) are used in place in HBM / L2, which lets a third environment walk the code with the other two.
struct VSmall3 : VSmall {
  static constexpr bool kItemsInPlace = true;
};
// ... and with the reference's default shape (128 players, 256 NPCs, 160^2 map, default record layout) folded in
struct VSmall3Std : VSmall3 {
  static constexpr bool kStd = true;
};
// ... four environments per CTA, NM_STEP4_THREADS threads each (P <= kThreads, P + N <= 2 * kThreads): a 4096-env
// tick is 1024 CTAs, seven full rounds of 148 SMs.  An environment gets 58 KB of shared memory (227 KB / 4), so the
// arrays that are rebuilt every tick and read off the critical path also go to the per-env workspace in HBM / L2
// (actions, task rows and accumulators, inventory lists, unique-event counts, window-scan results), the depleted-tile
// list is used in place, and the Move position index, the player list and the alive-player list share scratch arrays
// that are idle in the phases using them.  The NPC id hash stays: it is rebuilt and probed in the bookkeeping phase,
// which is on every tick's critical path (in HBM it cost 5 K cycles per env-tick late in an episode).
struct VSmall4 : VSmall3 {
  static constexpr int kThreads = NM_STEP4_THREADS;
  static constexpr bool kScratchInWs = true;
};
struct VSmall4Std : VSmall4 {
  static constexpr bool kStd = true;
};
struct VBig {
  static constexpr int kThreads = NM_BIG_THREADS;
  static constexpr int kRowsPerThread = 3;
  static constexpr int kChunkIters = 3;                 // <= 96 chunks
  static constexpr int kEvCap = NM_BIG_EV_CAP, kDeplCap = NM_BIG_DEPL_CAP, kNpcHash = 4096, kTblSlots = 8192;
  static constexpr bool kGlobalTables = true;           // tables are used where they live (HBM, served from L2)
  static constexpr bool kItemsInPlace = true;
  static constexpr bool kScratchInWs = false;
  static constexpr bool kStd = false;
  typedef StdShape5 Shape;
  typedef uint32_t tile_t;
  // row-major entity table, NM_BIG_ENT_STRIDE int16 per row: the columns of one entity share L2 sectors, and the
  // 31 observed columns are the first 62 bytes of the row, which is what the observation kernel copies out
  static __host__ __device__ __forceinline__ int ent_idx(int col, int row, int) { return row * NM_BIG_ENT_STRIDE + col; }
};
struct VBigStd : VBig {      // the configs[4] shape folded in
  static constexpr bool kStd = true;
};
// attack registrations: (round tag << kIdxBits) | index of the attack in the ordered list (< 4096 attacks per env)
constexpr int kIdxBits = 12;

enum { A_USE = 0, A_DESTROY, A_SELL_ITEM, A_SELL_PRICE, A_BUY, A_GIVE_ITEM, A_GIVE_TARGET, A_GOLD_AMT,
       A_GOLD_TARGET, A_ATT_STYLE, A_ATT_TARGET, A_MOVE, A_N };

template <class V>
struct Ctx {
  typedef typename V::tile_t tile_t;
  const NmParams *p;
  NmCfg<V::kStd> c;          // config vector (engine defaults folded in a *_std instantiation)
  int env, P, N, R, S, CAP, NINV;
  int16_t *ent, *item;
  uint32_t *map;            // 4-bit materials, 8 tiles per word
  tile_t *dlist;            // depleted tiles known at the start of the tick + the ones harvested during it (sc[17] = count)
  uint32_t *occ, *used, *fresh;
  uint16_t *inv;
  uint8_t *invn;
  int16_t *act;
  int8_t *npc_move;
  int16_t *npc_att;
  uint2 *ev;
  int *sc;            // shared scalars: [0] nev, [1] overflow, [2] n_danger, [3] next_npc_id, [4] npc_count
  int *duniq;
  unsigned short *npc_hash;   // open-addressing map NPC id -> row+1 (512 slots)
  int *task;                  // [P][4] pred, p0, p1, spare: the agent's task row for event folding
  int *acc;                   // [P][2] event-driven predicate accumulators
  int8_t *slow;               // [P] result of the window-scan predicates (-1 = not requested)
  const uint32_t *plist;      // alive players at the start of the step: row<<20 | r<<10 | c, ascending row
  int n_plist;
  const uint32_t *predraw;    // NPC-spawn draws computed in parallel: [attempt][8]
  uint64_t seed;
  int tick;
  int inj_lo, inj_hi;
};
#define ENT(col, row) ctx.ent[V::ent_idx((col), (row), ctx.R)]
#define ITM(col, row) ctx.item[(col) * ctx.CAP + (row)]

// one out-of-line copy of the draw (hash + injected-value lookup): it is called from ~16 sites and
// the step kernel is instruction-cache bound, not call bound
__device__ __forceinline__ uint32_t draw_impl(const uint64_t *inj_keys, const uint32_t *inj_vals, int lo, int hi,
                                           uint64_t seed, uint32_t tick, uint32_t site, uint32_t idx, uint32_t k) {
  if (hi > lo) {
    uint64_t key = nm_rng_key(tick, site, idx, k);
    hi -= 1;
    #pragma unroll 1
    while (lo <= hi) {
      int mid = (lo + hi) >> 1;
      uint64_t kk = inj_keys[mid];
      if (kk == key) return inj_vals[mid];
      if (kk < key) lo = mid + 1; else hi = mid - 1;
    }
  }
  return nm_hash_draw(seed, tick, site, idx, k);
}
template <class V>
__device__ __forceinline__ uint32_t draw(const Ctx<V> &ctx, uint32_t site, uint32_t idx, uint32_t k) {
  if (V::kStd) return nm_hash_draw(ctx.seed, (uint32_t)ctx.tick, site, idx, k);      // no injected draws in a *_std instantiation
  return draw_impl(ctx.p->inj_keys, ctx.p->inj_vals, ctx.inj_lo, ctx.inj_hi, ctx.seed, (uint32_t)ctx.tick, site, idx, k);
}

// ------------------------------------------------------------------ event ring ------
template <class V>
__device__ void emit(const Ctx<V> &ctx, int prow, int code, int type, int level, int number, int gold, int target) {
  int i = atomicAdd(&ctx.sc[0], 1);
  if (i >= ctx.p->ev_cap) { ctx.sc[1] = 1; return; }      // ev_cap = V::kEvCap (a test hook can lower it)
  // the target's id (players > 0, NPCs < 0) goes into the half of w1 its event leaves zero: number for LOOT_GOLD, gold
  // for SCORE_HIT, PLAYER_KILL and LOOT_ITEM.  fold_event reads neither there, and `code` is a constant at every call.
  if (code == EV_LOOT_GOLD) number = target;
  else if (target != 0) gold = target;
  // agent 16 bits | dense event 5 | item type / skill 5 | level 4 | target sign 2
  uint32_t w0 = (uint32_t)prow | ((uint32_t)nm_dense_event(code) << 16) | ((uint32_t)type << 21) |
                ((uint32_t)(level & 15) << 26) | (target > 0 ? (1u << 30) : 0u) | (target < 0 ? (1u << 31) : 0u);
  uint32_t w1 = (uint32_t)(uint16_t)number | ((uint32_t)(uint16_t)gold << 16);
  ctx.ev[i] = make_uint2(w0, w1);
}

// ----------------------------------------------------------- item / inventory -------
template <class V>
__device__ __forceinline__ bool row_used(const Ctx<V> &ctx, int row) { return (ctx.used[row >> 5] >> (row & 31)) & 1u; }
template <class V>
__device__ int item_alloc(const Ctx<V> &ctx) {          // lowest free row; sequential phases only
  int words = (ctx.CAP + 31) >> 5;
  #pragma unroll 1
  for (int w = 0; w < words; w++) {
    uint32_t freebits = ~ctx.used[w];
    if (freebits) {
      int row = (w << 5) + __ffs(freebits) - 1;
      if (row >= ctx.CAP) return -1;
      ctx.used[w] |= 1u << (row & 31);
      ctx.fresh[w] |= 1u << (row & 31);
      return row;
    }
  }
  return -1;
}
template <class V>
__device__ void inv_remove(const Ctx<V> &ctx, int owner_row, int row) {
  int n = ctx.invn[owner_row];
  uint16_t *l = ctx.inv + owner_row * ctx.NINV;
  #pragma unroll 1
  for (int i = 0; i < n; i++)
    if (l[i] == row) { l[i] = l[n - 1]; ctx.invn[owner_row] = (uint8_t)(n - 1); return; }
}
template <class V>
__device__ void inv_add(const Ctx<V> &ctx, int owner_row, int row) {
  int n = ctx.invn[owner_row];
  if (n < ctx.NINV) { ctx.inv[owner_row * ctx.NINV + n] = (uint16_t)row; ctx.invn[owner_row] = (uint8_t)(n + 1); }
}
template <class V>
__device__ int find_stack(const Ctx<V> &ctx, int owner_row, int type, int level, int exclude) {
  int n = ctx.invn[owner_row];
  const uint16_t *l = ctx.inv + owner_row * ctx.NINV;
  #pragma unroll 1
  for (int i = 0; i < n; i++) {
    int r = l[i];
    if (r != exclude && ITM(IS_TYPE, r) == type && ITM(IS_LEVEL, r) == level) return r;
  }
  return -1;
}
__device__ int equip_col(int type) {
  if (type == IT_HAT) return EA_EQ_HAT;
  if (type == IT_TOP) return EA_EQ_TOP;
  if (type == IT_BOTTOM) return EA_EQ_BOTTOM;
  if (it_weapon(type) || it_tool(type)) return EA_EQ_HELD;
  if (it_ammo(type)) return EA_EQ_AMMO;
  return -1;
}
// frees the row; the owner's list and equipment slot are fixed up (owner_row < 0: no owner)
template <class V>
__device__ void item_destroy(const Ctx<V> &ctx, int row) {
  int owner = ITM(IS_OWNER, row);
  if (owner > 0) {
    int orow = owner - 1;
    if (ITM(IS_EQUIPPED, row)) {
      int col = equip_col(ITM(IS_TYPE, row));
      if (col >= 0 && ENT(col, orow) == row + 1) ENT(col, orow) = 0;
    }
    inv_remove(ctx, orow, row);
  }
#pragma unroll
  for (int k = 0; k < IS_N; k++) ITM(k, row) = 0;
  atomicAnd(&ctx.used[row >> 5], ~(1u << (row & 31)));
}
// move an existing row into new_owner's inventory (ammo merges into an existing stack)
template <class V>
__device__ void inv_receive_existing(const Ctx<V> &ctx, int new_owner_row, int row) {
  int type = ITM(IS_TYPE, row);
  int old_owner = ITM(IS_OWNER, row);
  if (it_ammo(type)) {
    int st = find_stack(ctx, new_owner_row, type, ITM(IS_LEVEL, row), row);
    if (st >= 0) { ITM(IS_QUANTITY, st) = (int16_t)(ITM(IS_QUANTITY, st) + ITM(IS_QUANTITY, row)); item_destroy(ctx, row); return; }
  }
  if (old_owner > 0) inv_remove(ctx, old_owner - 1, row);
  ITM(IS_OWNER, row) = (int16_t)(new_owner_row + 1);
  inv_add(ctx, new_owner_row, row);
}
template <class V>
__device__ void inv_receive_new(const Ctx<V> &ctx, int owner_row, int type, int level, int qty) {
  if (it_ammo(type)) {
    int st = find_stack(ctx, owner_row, type, level, -1);
    if (st >= 0) { ITM(IS_QUANTITY, st) = (int16_t)(ITM(IS_QUANTITY, st) + qty); return; }
  }
  int row = item_alloc(ctx);
  if (row < 0) return;
  ITM(IS_TYPE, row) = (int16_t)type; ITM(IS_LEVEL, row) = (int16_t)level; ITM(IS_OWNER, row) = (int16_t)(owner_row + 1);
  ITM(IS_QUANTITY, row) = (int16_t)qty; ITM(IS_EQUIPPED, row) = 0; ITM(IS_PRICE, row) = 0; ITM(IS_LIST_TICK, row) = 0;
  inv_add(ctx, owner_row, row);
}
// item argument of a validated action: must still be the object the agent saw
template <class V>
__device__ int valid_item_ref(const Ctx<V> &ctx, int item_id, int owner) {
  if (item_id <= 0 || item_id > ctx.CAP) return -1;
  int row = item_id - 1;
  if (!row_used(ctx, row) || ((ctx.fresh[row >> 5] >> (row & 31)) & 1u)) return -1;
  if (owner && ITM(IS_OWNER, row) != owner) return -1;
  return row;
}

// -------------------------------------------------------------------- entities ------
template <class V>
__device__ __forceinline__ bool ent_alive(const Ctx<V> &ctx, int row) {
  return row >= 0 && ENT(EA_STATUS, row) == ES_ALIVE && ENT(EA_HEALTH, row) > 0;
}
template <class V>
__device__ int level_at_exp(const Ctx<V> &ctx, int exp) {
  int lmax = ctx.c[NC_LEVEL_MAX];
  if (exp >= ctx.c.p[NC_EXP_THRESH0 + lmax - 1]) return lmax;
  int lvl = 0;
  #pragma unroll 1
  while (lvl < lmax && exp >= ctx.c.p[NC_EXP_THRESH0 + lvl]) lvl++;
  return lvl;
}
template <class V>
__device__ void add_xp(const Ctx<V> &ctx, int row, int level_col, int skill_id, int xp) {
  int lmax = ctx.c[NC_LEVEL_MAX];
  int nexp = min(ENT(level_col + 1, row) + xp, ctx.c.p[NC_EXP_THRESH0 + lmax - 1]);
  ENT(level_col + 1, row) = (int16_t)nexp;
  int nl = level_at_exp(ctx, nexp);
  if (nl > ENT(level_col, row)) {
    ENT(level_col, row) = (int16_t)nl;
    if (row < ctx.P) emit(ctx, row, EV_LEVEL_UP, skill_id, nl, 0, 0, 0);
  }
}
template <class V>
__device__ int attack_level(const Ctx<V> &ctx, int row) {
  return max(ENT(EA_MELEE_LEVEL, row), max(ENT(EA_RANGE_LEVEL, row), ENT(EA_MAGE_LEVEL, row)));
}
template <class V>
__device__ int use_level(const Ctx<V> &ctx, int row, int type) {
  switch (type) {
    case IT_SPEAR: case IT_WHETSTONE: return ENT(EA_MELEE_LEVEL, row);
    case IT_BOW: case IT_ARROW: return ENT(EA_RANGE_LEVEL, row);
    case IT_WAND: case IT_RUNES: return ENT(EA_MAGE_LEVEL, row);
    case IT_ROD: return ENT(EA_FISHING_LEVEL, row);
    case IT_GLOVES: return ENT(EA_HERBALISM_LEVEL, row);
    case IT_PICKAXE: return ENT(EA_PROSPECTING_LEVEL, row);
    case IT_AXE: return ENT(EA_CARVING_LEVEL, row);
    case IT_CHISEL: return ENT(EA_ALCHEMY_LEVEL, row);
    default: {
      int l = 1;
      for (int col = EA_MELEE_LEVEL; col <= EA_ALCHEMY_LEVEL; col += 2) l = max(l, (int)ENT(col, row));
      return l;
    }
  }
}
// the tile map is packed 4 bits per tile (16 materials), tile i in bits 4*(i&7) of word i>>3
template <class V>
__device__ __forceinline__ int tile_i(const Ctx<V> &ctx, int i) { return (ctx.map[i >> 3] >> ((i & 7) * 4)) & 15; }
template <class V>
__device__ __forceinline__ int tile_at(const Ctx<V> &ctx, int r, int c) { return tile_i(ctx, r * ctx.S + c); }
// materials only ever change by one step (harvest: m -> m-1, respawn: m -> m+1) and never leave
// 0..15, so an atomic add on the word is an exact update of one nibble under concurrent writers
template <class V>
__device__ __forceinline__ void tile_dec(const Ctx<V> &ctx, int i) {      // harvest: the tile joins the depleted list
  atomicSub(&ctx.map[i >> 3], 1u << ((i & 7) * 4));
  const int k = atomicAdd(&ctx.sc[17], 1);
  if (k < V::kDeplCap) ctx.dlist[k] = (typename V::tile_t)i;
}
template <class V>
__device__ __forceinline__ void tile_inc(const Ctx<V> &ctx, int i) { atomicAdd(&ctx.map[i >> 3], 1u << ((i & 7) * 4)); }
template <class V>
__device__ __forceinline__ bool occ_get(const Ctx<V> &ctx, int r, int c) { int i = r * ctx.S + c; return (ctx.occ[i >> 5] >> (i & 31)) & 1u; }
template <class V>
__device__ __forceinline__ void occ_set(const Ctx<V> &ctx, int r, int c) { int i = r * ctx.S + c; atomicOr(&ctx.occ[i >> 5], 1u << (i & 31)); }
template <class V>
__device__ __forceinline__ void occ_clr(const Ctx<V> &ctx, int r, int c) { int i = r * ctx.S + c; atomicAnd(&ctx.occ[i >> 5], ~(1u << (i & 31))); }

// ------------------------------------------------------------------ harvesting ------
template <class V>
__device__ void process_drops(const Ctx<V> &ctx, int prow, int matl, int level_col, int skill_id) {
  int tool_type = 0, ammo = 0, weapon = 0, consumable = 0;
  switch (matl) {
    case MT_FISH: tool_type = IT_ROD; consumable = IT_RATION; break;
    case MT_HERB: tool_type = IT_GLOVES; consumable = IT_POTION; break;
    case MT_ORE: tool_type = IT_PICKAXE; ammo = IT_WHETSTONE; weapon = IT_WAND; break;
    case MT_TREE: tool_type = IT_AXE; ammo = IT_ARROW; weapon = IT_SPEAR; break;
    case MT_CRYSTAL: tool_type = IT_CHISEL; ammo = IT_RUNES; weapon = IT_BOW; break;
  }
  int level = 1;
  int held = ENT(EA_EQ_HELD, prow);
  if (held && ITM(IS_TYPE, held - 1) == tool_type) level = min(1 + ITM(IS_LEVEL, held - 1), ctx.c[NC_LEVEL_MAX]);
  int first = consumable ? consumable : ammo;
  if (ctx.invn[prow] < ctx.NINV) {
    inv_receive_new(ctx, prow, first, level, 1);
    emit(ctx, prow, EV_HARVEST_ITEM, first, level, 1, 0, 0);
  }
  if (weapon) {
    uint32_t u = draw(ctx, RS_HARVEST, (uint32_t)prow, (uint32_t)skill_id);
    if (u < (uint32_t)ctx.c[NC_WEAPON_DROP_THR] && ctx.invn[prow] < ctx.NINV) {
      inv_receive_new(ctx, prow, weapon, level, 1);
      emit(ctx, prow, EV_HARVEST_ITEM, weapon, level, 1, 0, 0);
    }
  }
  add_xp(ctx, prow, level_col, skill_id, consumable ? ctx.c[NC_XP_CONSUMABLE] : ctx.c[NC_XP_AMMO]);
}
template <class V>
__device__ bool tile_harvest(const Ctx<V> &ctx, int r, int c, int matl) {
  int i = r * ctx.S + c;
  if (tile_i(ctx, i) != matl) return false;
  tile_dec(ctx, i);
  return true;
}
// the id-ordered part of Player.update: anything that depletes a tile or allocates an item
template <class V>
__device__ void player_harvest(const Ctx<V> &ctx, int p) {
  int r = ENT(EA_ROW, p), c = ENT(EA_COL, p);
  if (tile_harvest(ctx, r, c, MT_FOILAGE)) {
    ENT(EA_FOOD, p) = (int16_t)min(ctx.c[NC_RES_BASE], ENT(EA_FOOD, p) + ctx.c[NC_RES_HARVEST_RESTORE]);
    emit(ctx, p, EV_EAT_FOOD, 0, 0, 0, 0, 0);
  }
  bool fish = false;
  fish |= tile_harvest(ctx, r - 1, c, MT_FISH);
  fish |= tile_harvest(ctx, r + 1, c, MT_FISH);
  fish |= tile_harvest(ctx, r, c - 1, MT_FISH);
  fish |= tile_harvest(ctx, r, c + 1, MT_FISH);
  if (fish) process_drops(ctx, p, MT_FISH, EA_FISHING_LEVEL, SK_FISHING);
  if (tile_harvest(ctx, r, c, MT_HERB)) process_drops(ctx, p, MT_HERB, EA_HERBALISM_LEVEL, SK_HERBALISM);
  if (tile_harvest(ctx, r, c, MT_ORE)) process_drops(ctx, p, MT_ORE, EA_PROSPECTING_LEVEL, SK_PROSPECTING);
  if (tile_harvest(ctx, r, c, MT_TREE)) process_drops(ctx, p, MT_TREE, EA_CARVING_LEVEL, SK_CARVING);
  if (tile_harvest(ctx, r, c, MT_CRYSTAL)) process_drops(ctx, p, MT_CRYSTAL, EA_ALCHEMY_LEVEL, SK_ALCHEMY);
}

// ---------------------------------------------------------------------- npc ai ------
template <class V>
__device__ bool valid_target(const Ctx<V> &ctx, int row, int targ_id, int rng) {
  if (targ_id <= 0 || targ_id > ctx.P) return false;      // NPCs only ever track players
  int t = targ_id - 1;
  if (!ent_alive(ctx, t)) return false;
  return nm_linf(ENT(EA_ROW, row), ENT(EA_COL, row), ENT(EA_ROW, t), ENT(EA_COL, t)) <= rng;
}
// first player met by the reference's ring scan (nmmo/systems/ai/utils.py closestTarget)
template <class V>
__device__ int closest_target(const Ctx<V> &ctx, int row, int rng) {
  int sr = ENT(EA_ROW, row), sc = ENT(EA_COL, row);
  {   // nothing but me inside the window? (11-bit row slices of the occupancy bitmap)
    unsigned any = 0;
    for (int rr = sr - rng; rr <= sr + rng; rr++) {
      int i0 = rr * ctx.S + sc - rng;
      unsigned bits = __funnelshift_r(ctx.occ[i0 >> 5], ctx.occ[(i0 >> 5) + 1], i0 & 31) & ((1u << (2 * rng + 1)) - 1);
      if (rr == sr && !ctx.c[NC_ALLOW_OCCUPIED]) bits &= ~(1u << rng);
      any |= bits;
    }
    if (!any) return 0;
  }
  int best = 0x7fffffff, best_id = 0;
  for (int k = 0; k < ctx.n_plist; k++) {
    uint32_t x = ctx.plist[k];
    int p = (int)(x >> 20);
    int dr = (int)((x >> 10) & 1023u) - sr, dc = (int)(x & 1023u) - sc;
    int d = max(nm_iabs(dr), nm_iabs(dc));
    if (d > rng) continue;
    int rk = 0x7fffffff;
    if (dc == -d) rk = min(rk, (dr + d) * 4 + 0);
    if (dc == d) rk = min(rk, (dr + d) * 4 + 1);
    if (dr == -d) rk = min(rk, (dc + d) * 4 + 2);
    if (dr == d) rk = min(rk, (dc + d) * 4 + 3);
    rk += d * 1024;
    if (rk < best) { best = rk; best_id = p + 1; }
  }
  return best_id;
}
// A* with the reference's 100-expansion budget; per-thread hash map + binary heap in local memory
// HN = node-table slots.  The search is first tried with a small table (cheap to clear; enough
// for the common open-ground chase) and repeated with the full-size table if it fills up; the
// result is identical either way.  Returns -2 when the table overflowed.
template <class V, int HN>
__device__ int astar_dir_t(const Ctx<V> &ctx, int sr, int sc, int gr, int gc) {
  const int CUTOFF = 100;
  uint16_t hk[HN]; uint8_t hcost[HN]; int8_t hback[HN];
  uint32_t heap[HN];
  if (sr == gr && sc == gc) return -1;
  for (int i = 0; i < HN; i++) hk[i] = 0;
  int n_nodes = 0;
  bool overflow = false;
  // nodes are keyed by their offset from the start tile (+128): the 100-expansion budget keeps the search within
  // 100 tiles of it, whatever the size of the map; a goal further away than that can never be found in the table
  const int kr = 128 - sr, kc = 128 - sc;
  auto slot_of = [&](int r, int c, bool insert) -> int {
    if ((unsigned)(r + kr) > 255u || (unsigned)(c + kc) > 255u) return -1;
    uint16_t key = (uint16_t)((((r + kr) << 8) | (c + kc)) + 1);
    int h = (int)((key * 40503u) >> 7) & (HN - 1);
        while (hk[h] != 0 && hk[h] != key) h = (h + 1) & (HN - 1);
    if (hk[h] == 0) {
      if (!insert) return -1;
      if (++n_nodes > (HN * 3) / 4) { overflow = true; return -1; }
      hk[h] = key; hcost[h] = 255; hback[h] = -1;
    }
    return h;
  };
  int hn = 0;
  auto push = [&](uint32_t x) {
    int i = hn++;
    heap[i] = x;
    while (i > 0) { int par = (i - 1) >> 1; if (heap[i] >= heap[par]) break; uint32_t t = heap[i]; heap[i] = heap[par]; heap[par] = t; i = par; }
  };
  auto pop = [&]() -> uint32_t {
    uint32_t top = heap[0];
    heap[0] = heap[--hn];
    int i = 0;
    for (;;) {
      int l = 2 * i + 1, r = l + 1, m = i;
      if (l < hn && heap[l] < heap[m]) m = l;
      if (r < hn && heap[r] < heap[m]) m = r;
      if (m == i) break;
      uint32_t t = heap[i]; heap[i] = heap[m]; heap[m] = t; i = m;
    }
    return top;
  };
  const int adr[4] = {-1, 1, 0, 0}, adc[4] = {0, 0, -1, 1};
  push((uint32_t)((128 << 8) | 128));
  { int s = slot_of(sr, sc, true); hcost[s] = 0; }
  int goal_r = gr, goal_c = gc, close_r = sr, close_c = sc;
  int close_h = nm_iabs(sr - gr) + nm_iabs(sc - gc), close_cost = close_h;
  int cutoff = CUTOFF;
  while (hn > 0) {
    cutoff--;
    if (cutoff <= 0) {
      int g = slot_of(gr, gc, false);
      if (!(g >= 0 && hback[g] >= 0)) { goal_r = close_r; goal_c = close_c; }
      break;
    }
    uint32_t cur = pop();
    int cr = (int)((cur >> 8) & 255) - kr, cc = (int)(cur & 255) - kc;
    if (cr == gr && cc == gc) break;
    int ccost = hcost[slot_of(cr, cc, false)];
        for (int k = 0; k < 4; k++) {
      int nr = cr + adr[k], nc = cc + adc[k];
      if (nr < 0 || nc < 0 || nr >= ctx.S || nc >= ctx.S) continue;
      if (nm_impassible(tile_at(ctx, nr, nc))) continue;
      int ncost = ccost + 1;
      int s = slot_of(nr, nc, true);
      if (overflow) return -2;
      if (hn >= HN - 1) return -2;
      if (hcost[s] == 255 || ncost < hcost[s]) {
        hcost[s] = (uint8_t)ncost;
        int h = nm_linf(gr, gc, nr, nc);
        int pri = ncost + h;
        if (h < close_h || (h == close_h && pri < close_cost)) { close_r = nr; close_c = nc; close_h = h; close_cost = pri; }
        push(((uint32_t)pri << 16) | (uint32_t)(((nr + kr) << 8) | (nc + kc)));
        hback[s] = (int8_t)k;
      }
    }
  }
  int r = goal_r, c = goal_c;
  for (;;) {
    int s = slot_of(r, c, false);
    if (s < 0 || hback[s] < 0) break;
    int pr = r - adr[hback[s]], pc = c - adc[hback[s]];
    if (pr == sr && pc == sc) break;
    r = pr; c = pc;
  }
  int dr = r - sr, dc = c - sc;
  if (dr == -1 && dc == 0) return 0;
  if (dr == 1 && dc == 0) return 1;
  if (dr == 0 && dc == 1) return 2;
  if (dr == 0 && dc == -1) return 3;
  return -1;
}
template <class V>
__device__ int astar_dir(const Ctx<V> &ctx, int sr, int sc, int gr, int gc) {
  int d = astar_dir_t<V, 64>(ctx, sr, sc, gr, gc);
  if (d == -2) d = astar_dir_t<V, 512>(ctx, sr, sc, gr, gc);
  return d;
}
template <class V>
__device__ void npc_decide(const Ctx<V> &ctx, int row) {
  int vis = ctx.c[NC_NPC_VISION];
  int n = row - ctx.P;
  uint32_t k = 0;
  ctx.npc_move[n] = -1;
  ctx.npc_att[n] = 0;
  int attacker = valid_target(ctx, row, ENT(EA_ATTACKER_ID, row), vis) ? ENT(EA_ATTACKER_ID, row) : 0;
  int target = ENT(EA_NPC_TARGET, row);
  if (!valid_target(ctx, row, target, vis)) target = 0;
  bool hunt = false;
  int type = ENT(EA_NPC_TYPE, row);
  if (type == 2) { if (attacker) { target = attacker; hunt = true; } }
  else if (type == 3) { if (!target) target = closest_target(ctx, row, vis); if (target) hunt = true; }
  ENT(EA_NPC_TARGET, row) = (int16_t)target;
  int r = ENT(EA_ROW, row), c = ENT(EA_COL, row);
  if (!hunt) {
    int start = nm_bounded(draw(ctx, RS_NPC_DECIDE, (uint32_t)row, k++), 4);
    int pick = start;
    for (int i = 0; i < 4; i++) {
      int d = (start + i) & 3;
      if (!nm_impassible(tile_at(ctx, r + c_dir_dr[d], c + c_dir_dc[d]))) { pick = d; break; }
    }
    ctx.npc_move[n] = (int8_t)pick;
    return;
  }
  int t = target - 1;
  int tr = ENT(EA_ROW, t), tc = ENT(EA_COL, t);
  int dist = nm_linf(r, c, tr, tc);
  if (dist == 0) ctx.npc_move[n] = (int8_t)nm_bounded(draw(ctx, RS_NPC_DECIDE, (uint32_t)row, k++), 4);
  else if (dist > 1) ctx.npc_move[n] = (int8_t)astar_dir(ctx, r, c, tr, tc);
  if (dist <= ctx.c[NC_REACH]) ctx.npc_att[n] = (int16_t)(t + 1);
}

// --------------------------------------------------------------------- actions ------
template <class V>
__device__ void act_use(const Ctx<V> &ctx, int p, int item_id) {
  int row = valid_item_ref(ctx, item_id, p + 1);
  if (row < 0) return;
  int type = ITM(IS_TYPE, row), level = ITM(IS_LEVEL, row);
  if (ITM(IS_PRICE, row) > 0 || level > use_level(ctx, p, type)) return;
  if (it_consumable(type)) {
    emit(ctx, p, EV_CONSUME_ITEM, type, level, ITM(IS_QUANTITY, row), 0, 0);
    int restore = ctx.c[NC_RESTORE_BASE] + level * ctx.c[NC_RESTORE_LEVEL];
    int base = ctx.c[NC_RES_BASE];
    if (type == IT_RATION) {
      ENT(EA_FOOD, p) = (int16_t)min(base, ENT(EA_FOOD, p) + restore);
      ENT(EA_WATER, p) = (int16_t)min(base, ENT(EA_WATER, p) + restore);
    } else ENT(EA_HEALTH, p) = (int16_t)min(base, ENT(EA_HEALTH, p) + restore);
    item_destroy(ctx, row);
    return;
  }
  int col = equip_col(type);
  if (col < 0) return;
  if (ITM(IS_EQUIPPED, row)) { ITM(IS_EQUIPPED, row) = 0; ENT(col, p) = 0; return; }
  int cur = ENT(col, p);
  if (cur) ITM(IS_EQUIPPED, cur - 1) = 0;
  ITM(IS_EQUIPPED, row) = 1; ENT(col, p) = (int16_t)(row + 1);
  emit(ctx, p, EV_EQUIP_ITEM, type, level, ITM(IS_QUANTITY, row), 0, 0);
}
template <class V>
__device__ void act_destroy(const Ctx<V> &ctx, int p, int item_id) {
  int row = valid_item_ref(ctx, item_id, p + 1);
  if (row < 0 || ITM(IS_EQUIPPED, row)) return;
  emit(ctx, p, EV_DESTROY_ITEM, ITM(IS_TYPE, row), ITM(IS_LEVEL, row), ITM(IS_QUANTITY, row), 0, 0);
  item_destroy(ctx, row);
}
template <class V>
__device__ void act_sell(const Ctx<V> &ctx, int p, int item_id, int price) {
  int row = valid_item_ref(ctx, item_id, p + 1);
  if (row < 0 || ITM(IS_EQUIPPED, row) || ITM(IS_PRICE, row)) return;
  ITM(IS_PRICE, row) = (int16_t)price; ITM(IS_LIST_TICK, row) = (int16_t)ctx.tick;
  emit(ctx, p, EV_LIST_ITEM, ITM(IS_TYPE, row), ITM(IS_LEVEL, row), ITM(IS_QUANTITY, row), price, 0);
}
template <class V>
__device__ void act_buy(const Ctx<V> &ctx, int p, int item_id) {
  int row = valid_item_ref(ctx, item_id, 0);
  if (row < 0) return;
  int owner = ITM(IS_OWNER, row), price = ITM(IS_PRICE, row);
  if (owner == 0 || price == 0) return;
  if (ENT(EA_GOLD, p) < price || owner == p + 1) return;
  int type = ITM(IS_TYPE, row), level = ITM(IS_LEVEL, row), qty = ITM(IS_QUANTITY, row);
  if (ctx.invn[p] >= ctx.NINV && !(it_ammo(type) && find_stack(ctx, p, type, level, -1) >= 0)) return;
  ITM(IS_PRICE, row) = 0; ITM(IS_LIST_TICK, row) = 0;
  inv_receive_existing(ctx, p, row);
  ENT(EA_GOLD, p) = (int16_t)(ENT(EA_GOLD, p) - price);
  ENT(EA_GOLD, owner - 1) = (int16_t)min(32767, ENT(EA_GOLD, owner - 1) + price);
  emit(ctx, p, EV_BUY_ITEM, type, level, qty, price, 0);
  emit(ctx, owner - 1, EV_EARN_GOLD, 0, 0, 0, price, 0);
}
template <class V>
__device__ void act_give(const Ctx<V> &ctx, int p, int item_id, int target_row1) {
  int row = valid_item_ref(ctx, item_id, p + 1);
  if (row < 0 || target_row1 <= 0) return;
  int t = target_row1 - 1;
  if (!ent_alive(ctx, t) || t == p) return;
  if (ITM(IS_EQUIPPED, row) || ITM(IS_PRICE, row)) return;
  if (ENT(EA_ROW, p) != ENT(EA_ROW, t) || ENT(EA_COL, p) != ENT(EA_COL, t)) return;
  int type = ITM(IS_TYPE, row), level = ITM(IS_LEVEL, row);
  if (ctx.invn[t] >= ctx.NINV && !(it_ammo(type) && find_stack(ctx, t, type, level, -1) >= 0)) return;
  emit(ctx, p, EV_GIVE_ITEM, type, level, ITM(IS_QUANTITY, row), 0, 0);
  inv_receive_existing(ctx, t, row);
}
template <class V>
__device__ void act_give_gold(const Ctx<V> &ctx, int p, int amount, int target_row1) {
  if (target_row1 <= 0) return;
  int t = target_row1 - 1;
  if (!ent_alive(ctx, t) || t == p) return;
  if (ENT(EA_ROW, p) != ENT(EA_ROW, t) || ENT(EA_COL, p) != ENT(EA_COL, t)) return;
  if (!(amount > 0 && ENT(EA_GOLD, p) > 0)) return;
  amount = min(amount, (int)ENT(EA_GOLD, p));
  ENT(EA_GOLD, p) = (int16_t)(ENT(EA_GOLD, p) - amount);
  ENT(EA_GOLD, t) = (int16_t)min(32767, ENT(EA_GOLD, t) + amount);
  emit(ctx, p, EV_GIVE_GOLD, 0, 0, 0, amount, 0);
}
// pure part of combat.attack / Attack.call: validity and damage, no side effects
template <class V>
__device__ bool attack_compute(const Ctx<V> &ctx, int a, int style, int t, int &dmg, bool &ammo_out) {
  const NmCfg<V::kStd> c = ctx.c;
  bool a_player = a < ctx.P, b_player = t < ctx.P;
  if (a_player && b_player && ENT(EA_TIME_ALIVE, t) < c[NC_SPAWN_IMMUNITY]) return false;
  if (!ent_alive(ctx, t)) return false;
  if (nm_linf(ENT(EA_ROW, a), ENT(EA_COL, a), ENT(EA_ROW, t), ENT(EA_COL, t)) > c[NC_REACH]) return false;
  int ex0 = ENT(EA_MELEE_EXP, t), ex1 = ENT(EA_RANGE_EXP, t), ex2 = ENT(EA_MAGE_EXP, t);
  int num = 1, den = 1;
  if (!(ex0 == ex1 && ex1 == ex2)) {
    int idx = 0, best = ex0;
    if (ex1 > best) { best = ex1; idx = 1; }
    if (ex2 > best) { best = ex2; idx = 2; }
    int weak = idx == 0 ? 2 : (idx == 1 ? 0 : 1);
    if (style == weak) { num = c[NC_WEAK_NUM]; den = c[NC_WEAK_DEN]; }
  }
  int lcol = EA_MELEE_LEVEL + 2 * style;
  int offense = c[NC_BASE_DAMAGE] + c[NC_LEVEL_DAMAGE] * ENT(lcol, a);
  int defense = c[NC_BASE_DEFENSE] + c[NC_LEVEL_DEFENSE] * ENT(lcol, t);
  ammo_out = false;
  if (a_player) {
    for (int s = EA_EQ_HAT; s <= EA_EQ_AMMO; s++) {
      int it = ENT(s, a);
      if (it) offense += item_attack(c, ITM(IS_TYPE, it - 1), ITM(IS_LEVEL, it - 1), style);
    }
    int am = ENT(EA_EQ_AMMO, a);
    if (am && item_attack(c, ITM(IS_TYPE, am - 1), ITM(IS_LEVEL, am - 1), style) > 0) ammo_out = ITM(IS_QUANTITY, am - 1) - 1 <= 0;
  } else offense += ENT(EA_NPC_OFFENSE, a);
  if (b_player) {
    for (int s = EA_EQ_HAT; s <= EA_EQ_AMMO; s++) {
      int it = ENT(s, t);
      if (it) defense += item_defense(c, ITM(IS_TYPE, it - 1), ITM(IS_LEVEL, it - 1));
    }
  } else defense += ENT(EA_NPC_DEFENSE, t);
  int min_dmg = (c[NC_MINDMG_NUM] * offense) / c[NC_MINDMG_DEN];
  dmg = (num * (offense - defense)) / den;
  dmg = max(min_dmg, dmg);
  dmg = min(dmg, (int)ENT(EA_HEALTH, t));
  return true;
}
// side effects of one attack whose damage is known (attacker a, target row t)
template <class V>
__device__ void attack_apply(const Ctx<V> &ctx, int a, int style, int t, int dmg) {
  const NmCfg<V::kStd> c = ctx.c;
  bool a_player = a < ctx.P, b_player = t < ctx.P;
  int a_id = ENT(EA_ID, a), b_id = ENT(EA_ID, t);
  int lcol = EA_MELEE_LEVEL + 2 * style;
  ENT(EA_ATTACKER_ID, t) = (int16_t)a_id;
  if (a_player) {
    int am = ENT(EA_EQ_AMMO, a);
    if (am && item_attack(c, ITM(IS_TYPE, am - 1), ITM(IS_LEVEL, am - 1), style) > 0) {
      int q = ITM(IS_QUANTITY, am - 1) - 1;
      ITM(IS_QUANTITY, am - 1) = (int16_t)q;
      if (q <= 0) item_destroy(ctx, am - 1);
    }
  }
  if (a_player) emit(ctx, a, EV_SCORE_HIT, SK_MELEE + style, 0, dmg, 0, b_id);
  ENT(EA_DMG_INFLICTED, a) = (int16_t)min(32767, ENT(EA_DMG_INFLICTED, a) + dmg);
  if (a_player) add_xp(ctx, a, lcol, SK_MELEE + style, c[NC_XP_COMBAT]);
  ENT(EA_DMG_RECEIVED, t) = (int16_t)min(32767, ENT(EA_DMG_RECEIVED, t) + dmg);
  ENT(EA_DAMAGE, t) = (int16_t)dmg;
  ENT(EA_HEALTH, t) = (int16_t)(ENT(EA_HEALTH, t) - dmg);
  if (style == 2 && dmg > 0) ENT(EA_FREEZE, t) = (int16_t)c[NC_FREEZE_TIME];
  ENT(EA_LATEST_COMBAT_TICK, a) = (int16_t)(ctx.tick + 1);
  ENT(EA_LATEST_COMBAT_TICK, t) = (int16_t)(ctx.tick + 1);
  if (ENT(EA_HEALTH, t) > 0) return;
  if (a_player) emit(ctx, a, EV_PLAYER_KILL, 0, attack_level(ctx, t), 0, 0, b_id);
  int tg = ENT(EA_GOLD, t);
  if (tg > 0) {
    ENT(EA_GOLD, a) = (int16_t)min(32767, ENT(EA_GOLD, a) + tg);
    if (a_player) emit(ctx, a, EV_LOOT_GOLD, 0, 0, 0, tg, b_id);
    ENT(EA_GOLD, t) = 0;
  }
  if (b_player) {
    // the victim's items in table-row order: unlist, then loot (player killer) or destroy
    int n = ctx.invn[t];
    uint16_t rows[16];
    #pragma unroll 1
    for (int i = 0; i < n; i++) rows[i] = ctx.inv[t * ctx.NINV + i];
    #pragma unroll 1
    for (int i = 1; i < n; i++) { uint16_t x = rows[i]; int j = i - 1; while (j >= 0 && rows[j] > x) { rows[j + 1] = rows[j]; j--; } rows[j + 1] = x; }
    #pragma unroll 1
    for (int i = 0; i < n; i++) {
      int row = rows[i];
      ITM(IS_PRICE, row) = 0; ITM(IS_LIST_TICK, row) = 0;
      if (ITM(IS_EQUIPPED, row)) { int col = equip_col(ITM(IS_TYPE, row)); if (col >= 0) ENT(col, t) = 0; ITM(IS_EQUIPPED, row) = 0; }
      if (a_player && ctx.invn[a] < ctx.NINV) {
        emit(ctx, a, EV_LOOT_ITEM, ITM(IS_TYPE, row), ITM(IS_LEVEL, row), ITM(IS_QUANTITY, row), 0, b_id);
        inv_receive_existing(ctx, a, row);
      } else item_destroy(ctx, row);
    }
  } else if (a_player) {
    int lvl = attack_level(ctx, t);
    int drops[2] = {ENT(EA_NPC_DROP_ARMOR, t), ENT(EA_NPC_DROP_TOOL, t)};
    for (int k2 = 0; k2 < 2; k2++)
      if (ctx.invn[a] < ctx.NINV) {
        inv_receive_new(ctx, a, drops[k2], lvl, 1);
        emit(ctx, a, EV_LOOT_ITEM, drops[k2], lvl, 1, 0, b_id);
      }
  }
}
template <class V>
__device__ void act_move(const Ctx<V> &ctx, int row, int dir, bool use_occ) {
  if (dir < 0 || dir > 3) return;
  if (ENT(EA_FREEZE, row) > 0) return;
  int r = ENT(EA_ROW, row), c = ENT(EA_COL, row);
  int nr = r + c_dir_dr[dir], nc = c + c_dir_dc[dir];
  if (nm_impassible(tile_at(ctx, nr, nc))) return;
  if (use_occ) {
    if (occ_get(ctx, nr, nc)) return;
    occ_clr(ctx, r, c); occ_set(ctx, nr, nc);
  }
  ENT(EA_ROW, row) = (int16_t)nr; ENT(EA_COL, row) = (int16_t)nc;
  if (row < ctx.P) {
    int half = ctx.S / 2;
    int progress = ctx.c[NC_MAP_CENTER] / 2 - nm_linf(half, half, nr, nc);
    if (progress > ENT(EA_EXPLORATION, row)) {
      ENT(EA_EXPLORATION, row) = (int16_t)progress;
      emit(ctx, row, EV_GO_FARTHEST, 0, 0, progress, 0, 0);
    }
  }
}

// ------------------------------------------------------------------ npc spawning ----
template <class V>
__device__ int border_dist(const Ctx<V> &ctx, int r, int c) {
  int b = ctx.c[NC_MAP_BORDER], ce = ctx.c[NC_MAP_CENTER];
  return min(min(r - b, ce + b - r - 1), min(c - b, ce + b - c - 1));
}
// NPCManager.spawn, split: the accept / reject logic of the (up to 25, at most 32) attempts is replayed by warp 0 and
// records the accepted ones; the rows are then filled in by one thread each.
// While the danger stack is not empty an attempt's position depends on how many attempts were accepted before it
// (the stack is popped per accept), so lane 0 walks those attempts one by one.  Once the stack is empty -- always, until
// NPCs start dying -- the positions of all remaining attempts are known up front: one lane per attempt checks its tile,
// an attempt loses to an earlier valid attempt on the same tile (match.any), a ballot prefix gives the n-th accepted
// attempt the n-th free row and cuts at the population limit.  Same result as the one-by-one walk.
template <class V>
__device__ int npc_spawn_decide(const Ctx<V> &ctx, uint32_t *dec, const int *free_rows, const int *dng, int lane) {       // warp 0
  const NmCfg<V::kStd> c = ctx.c;
  const int b = c[NC_MAP_BORDER], ce = c[NC_MAP_CENTER];
  const int attempts = min(c[NC_NPC_SPAWN_ATTEMPTS], 32);
  auto npc_type_at = [&](int d) -> int {
    if (200 * d >= c[NC_NPC_AGGR_PCT] * ce) return 3;
    if (200 * d >= c[NC_NPC_NEUT_PCT] * ce) return 2;
    if (200 * d >= c[NC_NPC_PASS_PCT] * ce) return 1;
    return 0;
  };
  int count = ctx.sc[4], n = 0, att = 0;
  const int nd0 = ctx.sc[2];
  int nd = nd0;
  if (lane == 0) {
    #pragma unroll 1
    for (; att < attempts && nd > 0; att++) {
      if (count >= ctx.N) break;
      // the n-th accepted spawn takes the n-th free row (the reference scans for the first free slot)
      const int scan = free_rows[n];
      const int d0 = dng[nd0 - nd];
      const int mid = ce / 2, max_off = mid - d0;
      const int offset = mid + b + nm_bounded(ctx.predraw[att * 8 + 0], 2 * max_off) - max_off;
      const int side = nm_bounded(ctx.predraw[att * 8 + 1], 4);
      int r, cc;
      if (side == 0) { r = b + d0; cc = offset; }
      else if (side == 1) { r = b + ce - d0 - 1; cc = offset; }
      else if (side == 2) { cc = b + d0; r = offset; }
      else { cc = b + ce - d0 - 1; r = offset; }
      if (nm_impassible(tile_at(ctx, r, cc))) continue;
      if (!c[NC_ALLOW_OCCUPIED] && occ_get(ctx, r, cc)) continue;
      const int d = border_dist(ctx, r, cc), type = npc_type_at(d);
      if (!type) continue;
      uint32_t *q = dec + n * 8;
      q[0] = (uint32_t)scan; q[1] = (uint32_t)r; q[2] = (uint32_t)cc; q[3] = (uint32_t)d; q[4] = (uint32_t)type;
      q[5] = (uint32_t)att; q[6] = (uint32_t)ctx.sc[3];
      ctx.sc[3]--;
      ENT(EA_STATUS, scan) = ES_ALIVE;
      occ_set(ctx, r, cc);
      count++; n++; nd--;
    }
  }
  __syncwarp();
  att = __shfl_sync(0xffffffffu, att, 0); n = __shfl_sync(0xffffffffu, n, 0);
  count = __shfl_sync(0xffffffffu, count, 0); nd = __shfl_sync(0xffffffffu, nd, 0);
  int n_b = 0;
  if (nd == 0 && count < ctx.N && att < attempts) {      // (warp-uniform) the remaining attempts, one per lane
    const int my_att = att + lane;
    const bool active = my_att < attempts;
    int r = 0, cc = 0, d = 0, type = 0;
    bool valid = false;
    if (active) {
      r = b + nm_bounded(ctx.predraw[my_att * 8 + 0], ce);
      cc = b + nm_bounded(ctx.predraw[my_att * 8 + 1], ce);
      valid = !nm_impassible(tile_at(ctx, r, cc)) && (c[NC_ALLOW_OCCUPIED] || !occ_get(ctx, r, cc));
      if (valid) { d = border_dist(ctx, r, cc); type = npc_type_at(d); valid = type != 0; }
    }
    const unsigned lt = (1u << lane) - 1u;
    const unsigned vm = __ballot_sync(0xffffffffu, valid);
    const unsigned same = __match_any_sync(0xffffffffu, valid ? r * ctx.S + cc : -1 - lane);
    const bool acc = valid && (c[NC_ALLOW_OCCUPIED] || !(same & vm & lt));
    const unsigned am = __ballot_sync(0xffffffffu, acc);
    const int rank = __popc(am & lt), limit = ctx.N - count, sc3 = ctx.sc[3];
    n_b = min(__popc(am), limit);
    __syncwarp();
    if (acc && rank < limit) {
      const int slot = n + rank, scan = free_rows[slot];
      uint32_t *q = dec + slot * 8;
      q[0] = (uint32_t)scan; q[1] = (uint32_t)r; q[2] = (uint32_t)cc; q[3] = (uint32_t)d; q[4] = (uint32_t)type;
      q[5] = (uint32_t)my_att; q[6] = (uint32_t)(sc3 - rank);
      ENT(EA_STATUS, scan) = ES_ALIVE;
      occ_set(ctx, r, cc);
    }
    if (lane == 0) ctx.sc[3] = sc3 - n_b;
  }
  if (lane == 0) ctx.sc[2] = nd;
  return n + n_b;
}
template <class V>
__device__ void npc_spawn_fill(const Ctx<V> &ctx, const uint32_t *q) {
  const NmCfg<V::kStd> c = ctx.c;
  int ce = c[NC_MAP_CENTER];
  int row = (int)q[0], r = (int)q[1], cc = (int)q[2], d = (int)q[3], type = (int)q[4], att = (int)q[5];
  int style = nm_bounded(ctx.predraw[att * 8 + 2], 3);
  int level = (2 * d * (c[NC_NPC_LEVEL_MAX] - c[NC_NPC_LEVEL_MIN])) / ce + c[NC_NPC_LEVEL_MIN];
  int frac = (int)(ctx.predraw[att * 8 + 3] >> 16);
  int lvl_fp = level * 65536 - frac;
  int armor = IT_HAT + nm_bounded(ctx.predraw[att * 8 + 4], 3);
  int tool = IT_ROD + nm_bounded(ctx.predraw[att * 8 + 5], 5);
  for (int col = 0; col < EA_N; col++) if (col != EA_STATUS) ENT(col, row) = 0;
  ENT(EA_ID, row) = (int16_t)(int)q[6];
  ENT(EA_NPC_TYPE, row) = (int16_t)type; ENT(EA_ROW, row) = (int16_t)r; ENT(EA_COL, row) = (int16_t)cc;
  ENT(EA_GOLD, row) = (int16_t)level;
  ENT(EA_HEALTH, row) = (int16_t)c[NC_RES_BASE]; ENT(EA_FOOD, row) = (int16_t)c[NC_RES_BASE]; ENT(EA_WATER, row) = (int16_t)c[NC_RES_BASE];
  for (int s = 0; s < 3; s++) ENT(EA_MELEE_LEVEL + 2 * s, row) = 1;
  ENT(EA_MELEE_LEVEL + 2 * style, row) = (int16_t)level;
  ENT(EA_MELEE_EXP + 2 * style, row) = (int16_t)c.p[NC_EXP_THRESH0 + level - 1];
  ENT(EA_ITEM_LEVEL, row) = (int16_t)((5LL * lvl_fp) >> 16);
  ENT(EA_NPC_STYLE, row) = (int16_t)style; ENT(EA_NPC_DANGER, row) = (int16_t)d;
  ENT(EA_NPC_OFFENSE, row) = (int16_t)(c[NC_NPC_BASE_DAMAGE] + (int)(((int64_t)lvl_fp * c[NC_NPC_LEVEL_DAMAGE]) >> 16));
  ENT(EA_NPC_DEFENSE, row) = (int16_t)(c[NC_NPC_BASE_DEFENSE] + (int)(((int64_t)lvl_fp * c[NC_NPC_LEVEL_DEFENSE]) >> 16));
  ENT(EA_NPC_DROP_ARMOR, row) = (int16_t)armor; ENT(EA_NPC_DROP_TOOL, row) = (int16_t)tool;
}

// ------------------------------------------------------------------------ tasks -----
__device__ double clip01(double x) { return x > 1.0 ? 1.0 : (x < 0.0 ? 0.0 : x); }
template <class V>
__device__ bool sees_tile(const Ctx<V> &ctx, int p, int matl) {
  const int vis = ctx.c[NC_VISION], r = ENT(EA_ROW, p), c = ENT(EA_COL, p);
  #pragma unroll 1
  for (int dr = -vis; dr <= vis; dr++)
    #pragma unroll 1
    for (int dc = -vis; dc <= vis; dc++)
      if (tile_at(ctx, r + dr, c + dc) == matl) return true;
  return false;
}
// is an entity with id in [lo, hi] among the first n_ent table rows inside p's vision window?
template <class V>
__device__ bool sees_ids(const Ctx<V> &ctx, int p, int lo, int hi) {
  const int vis = ctx.c[NC_VISION], r = ENT(EA_ROW, p), c = ENT(EA_COL, p);
  int seen = 0;
  #pragma unroll 1
  for (int row = 0; row < ctx.R && seen < ctx.p->L.n_ent; row++) {
    if (ENT(EA_STATUS, row) != ES_ALIVE) continue;
    if (nm_iabs(ENT(EA_ROW, row) - r) > vis || nm_iabs(ENT(EA_COL, row) - c) > vis) continue;
    seen++;
    const int id = ENT(EA_ID, row);
    if (id >= lo && id <= hi) return true;
  }
  return false;
}
// Team subjects and named targets (nm_task_flag).  Teams are consecutive id ranges of NC_TEAM_SIZE players; a
// TF_TEAM task is evaluated over the alive members of the assignee's team (every member holds the same task and
// computes the same value); TF_RELATIVE_TARGET resolves "left/right team (leader)" from the assignee's team.
template <class V>
__device__ double eval_team_predicate(const Ctx<V> &ctx, int p, int pred, int p0, int p1, int p2, int flags, bool &handled) {
  const int ts = max(1, ctx.c[NC_TEAM_SIZE]), nt = (ctx.P + ts - 1) / ts, team = p / ts;
  const int m0 = (flags & TF_TEAM) ? team * ts : p, m1 = (flags & TF_TEAM) ? min(ctx.P, m0 + ts) : p + 1;      // subject rows
  int lo = p0, hi = pred == TP_CAN_SEE_AGENT ? p0 : p1;                                                          // target ids
  int t0 = m0, t1 = m1;                                                                                          // target rows (AllDead)
  if (flags & TF_RELATIVE_TARGET) {
    const int tt = (((team + p0) % nt) + nt) % nt;
    t0 = tt * ts; t1 = min(ctx.P, t0 + ts);
    if (pred == TP_CAN_SEE_AGENT || (pred == TP_ALL_DEAD && p1 == 1)) t1 = t0 + 1;                               // the leader
    lo = t0 + 1; hi = t1;
  }
  handled = true;
  int num = 0, den = 1;
  switch (pred) {
    case TP_CAN_SEE_TILE:
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (ent_alive(ctx, m) && sees_tile(ctx, m, p0)) return 1.0;
      return 0.0;
    case TP_CAN_SEE_AGENT: case TP_CAN_SEE_GROUP:
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (ent_alive(ctx, m) && sees_ids(ctx, m, lo, hi)) return 1.0;
      return 0.0;
    case TP_OCCUPY_TILE:
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (ent_alive(ctx, m) && ENT(EA_ROW, m) == p0 && ENT(EA_COL, m) == p1) return 1.0;
      return 0.0;
    case TP_STAY_ALIVE:
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (!ent_alive(ctx, m)) return 0.0;
      return 1.0;
    case TP_ALL_DEAD:
      #pragma unroll 1
      for (int m = t0; m < t1; m++) num += ent_alive(ctx, m) ? 0 : 1;
      den = t1 - t0; break;
    case TP_ALL_MEMBERS_WITHIN_RANGE: {
      int r0 = 1 << 20, r1 = -1, c0 = 1 << 20, c1 = -1;
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (ent_alive(ctx, m)) {
        r0 = min(r0, (int)ENT(EA_ROW, m)); r1 = max(r1, (int)ENT(EA_ROW, m)); c0 = min(c0, (int)ENT(EA_COL, m)); c1 = max(c1, (int)ENT(EA_COL, m));
      }
      return (r1 - r0 <= p0 && c1 - c0 <= p0) ? 1.0 : 0.0;
    }
    case TP_DISTANCE_TRAVELED:
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (ent_alive(ctx, m)) num += nm_linf(ENT(EA_ROW, m), ENT(EA_COL, m), ENT(EA_SPAWN_ROW, m), ENT(EA_SPAWN_COL, m));
      den = p0; break;
    case TP_HOARD_GOLD:
      #pragma unroll 1
      for (int m = m0; m < m1; m++) if (ent_alive(ctx, m)) num += ENT(EA_GOLD, m);
      den = p0; break;
    case TP_COUNT_EVENT: case TP_SCORE_HIT: case TP_EARN_GOLD: case TP_SPEND_GOLD: case TP_MAKE_PROFIT: case TP_CONSUME_ITEM:
    case TP_HARVEST_ITEM: case TP_LIST_ITEM: case TP_BUY_ITEM: case TP_DEFEAT_ENTITY: {
      // the event-driven accumulators of every member (each counts its own events for the shared task)
      #pragma unroll 1
      for (int m = m0; m < m1; m++) num += ctx.acc[m * 2] - (pred == TP_MAKE_PROFIT ? ctx.acc[m * 2 + 1] : 0);
      den = (pred == TP_COUNT_EVENT || pred == TP_SCORE_HIT) ? p1 : (pred == TP_EARN_GOLD || pred == TP_SPEND_GOLD || pred == TP_MAKE_PROFIT) ? p0 : p2;
      break;
    }
    default: handled = false; return 0.0;      // evaluated on the agent itself
  }
  if (den > 0) { if (num <= 0) return 0.0; if (num >= den) return 1.0; }
  return clip01((double)num / (double)den);
}
template <class V>
__device__ double eval_predicate(const Ctx<V> &ctx, int p, int pred, int p0, int p1, int p2, int acc0, int acc1) {
  int vis = ctx.c[NC_VISION];
  // Ratio predicates only pick (num, den) here; the one f64 division sits behind the switch, and is skipped when
  // the clipped result is known without it (nothing counted yet, or the goal already reached).
  int num = 0, den = 1;
  switch (pred) {
    case TP_TICK_GE: num = ctx.tick; den = p0; break;
    case TP_COUNT_EVENT: case TP_SCORE_HIT: num = acc0; den = p1; break;
    case TP_CAN_SEE_TILE: {
      if (ctx.slow[p] >= 0) return (double)ctx.slow[p];
      int r = ENT(EA_ROW, p), c = ENT(EA_COL, p);
      #pragma unroll 1
      for (int dr = -vis; dr <= vis; dr++) for (int dc = -vis; dc <= vis; dc++)
        if (tile_at(ctx, r + dr, c + dc) == p0) return 1.0;
      return 0.0;
    }
    case TP_CAN_SEE_AGENT: case TP_CAN_SEE_GROUP: {
      // visible = among the first n_ent table rows inside the vision window
      if (ctx.slow[p] >= 0) return (double)ctx.slow[p];
      int lo = p0, hi = pred == TP_CAN_SEE_AGENT ? p0 : p1;
      int r = ENT(EA_ROW, p), c = ENT(EA_COL, p), seen = 0;
      #pragma unroll 1
      for (int row = 0; row < ctx.R && seen < ctx.p->L.n_ent; row++) {
        if (ENT(EA_STATUS, row) != ES_ALIVE) continue;
        if (nm_iabs(ENT(EA_ROW, row) - r) > vis || nm_iabs(ENT(EA_COL, row) - c) > vis) continue;
        seen++;
        int id = ENT(EA_ID, row);
        if (id >= lo && id <= hi) return 1.0;
      }
      return 0.0;
    }
    case TP_OCCUPY_TILE: return (ENT(EA_ROW, p) == p0 && ENT(EA_COL, p) == p1) ? 1.0 : 0.0;
    case TP_ATTAIN_SKILL:
      if (p1 <= 1) return 1.0;
      num = ENT(EA_MELEE_LEVEL + 2 * (p0 - 1), p) - 1; den = p1 - 1; break;
    case TP_GAIN_EXPERIENCE: num = min((int)ENT(EA_MELEE_EXP + 2 * (p0 - 1), p), p1); den = p1; break;
    case TP_EQUIP_ITEM: {
      int k = 0;
      #pragma unroll 1
      for (int i = 0; i < ctx.invn[p]; i++) { int r = ctx.inv[p * ctx.NINV + i];
        if (ITM(IS_TYPE, r) == p0 && ITM(IS_LEVEL, r) >= p1 && ITM(IS_EQUIPPED, r)) k++; }
      num = k; den = 1; break;
    }
    case TP_HOARD_GOLD: num = ENT(EA_GOLD, p); den = p0; break;
    case TP_EARN_GOLD: case TP_SPEND_GOLD: num = acc0; den = p0; break;
    case TP_MAKE_PROFIT: num = acc0 - acc1; den = p0; break;
    case TP_INVENTORY_SPACE_GE: return (ctx.NINV - ctx.invn[p] >= p0) ? 1.0 : 0.0;
    case TP_OWN_ITEM: {
      int s = 0;
      #pragma unroll 1
      for (int i = 0; i < ctx.invn[p]; i++) { int r = ctx.inv[p * ctx.NINV + i];
        if (ITM(IS_TYPE, r) == p0 && ITM(IS_LEVEL, r) >= p1) s += ITM(IS_QUANTITY, r); }
      num = s; den = p2; break;
    }
    case TP_CONSUME_ITEM: case TP_HARVEST_ITEM: case TP_LIST_ITEM: case TP_BUY_ITEM: case TP_DEFEAT_ENTITY:
      num = acc0; den = p2; break;
    case TP_FULLY_ARMED: {
      int need[5] = {IT_SPEAR + (p0 - 1), IT_WHETSTONE + (p0 - 1), IT_HAT, IT_TOP, IT_BOTTOM}, k = 0;
      #pragma unroll 1
      for (int j = 0; j < 5; j++)
        #pragma unroll 1
        for (int i = 0; i < ctx.invn[p]; i++) { int r = ctx.inv[p * ctx.NINV + i];
          if (ITM(IS_TYPE, r) == need[j] && ITM(IS_LEVEL, r) >= p1 && ITM(IS_EQUIPPED, r)) { k++; break; } }
      return k == 5 ? 1.0 : 0.0;
    }
    case TP_STAY_ALIVE: return ENT(EA_HEALTH, p) > 0 ? 1.0 : 0.0;
    case TP_DISTANCE_TRAVELED:
      num = nm_linf(ENT(EA_ROW, p), ENT(EA_COL, p), ENT(EA_SPAWN_ROW, p), ENT(EA_SPAWN_COL, p)); den = p0; break;
    case TP_ALL_DEAD: return ENT(EA_HEALTH, p) > 0 ? 0.0 : 1.0;
    case TP_ALL_MEMBERS_WITHIN_RANGE: return 1.0;
    default: return 0.0;
  }
  if (den > 0) {      // same value as the clipped quotient: <= 0 clips to 0.0, >= 1 clips to 1.0
    if (num <= 0) return 0.0;
    if (num >= den) return 1.0;
  }
  return clip01((double)num / (double)den);
}

// whole value of a flagged task (team subject and/or named target), incl. the second predicate and the combinator
// (measured: as a real call -- __noinline__ -- its mere presence costs the step kernel 22 %, inlined < 1 %)
template <class V>
__device__ __forceinline__ double flagged_task_value(const Ctx<V> &ctx, int p, int4 ta, int4 tb, int4 tc, int acc0, int acc1) {
  const int flags = tb.x;
  auto one = [&](int pred, int p0, int p1, int p2, int a0, int a1) -> double {
    bool handled;
    const double v = eval_team_predicate(ctx, p, pred, p0, p1, p2, flags, handled);
    return handled ? v : eval_predicate(ctx, p, pred, p0, p1, p2, a0, a1);
  };
  double v = one(ta.x, ta.y, ta.z, ta.w, acc0, acc1);
  if (tb.w == 1) v = v * one(tb.y, tb.z, tc.x, tc.y, 0, 0);
  else if (tb.w == 2)
    v = __dadd_rn(__dmul_rn(__ddiv_rn((double)tc.z, 1000.0), v), __dmul_rn(__ddiv_rn((double)tc.w, 1000.0), one(tb.y, tb.z, tc.x, tc.y, 0, 0)));
  return v;
}

// fold one event into the agent's accumulators (process_event_log / count_unique_events /
// event-driven predicates), order-free
template <class V>
__device__ void fold_event(const Ctx<V> &ctx, uint2 e) {
  int agent = e.x & 0xffff, de = (e.x >> 16) & 31, type = (e.x >> 21) & 31, level = (e.x >> 26) & 15;
  bool tpos = (e.x >> 30) & 1, tneg = (e.x >> 31) & 1;
  int number = (int)(int16_t)(e.y & 0xFFFF), gold = (int)(int16_t)(e.y >> 16);
  size_t a = (size_t)ctx.env * ctx.P + agent;
  int32_t *st = ctx.p->stats + a * ST_N;
  atomicAdd(&st[ST_EVT0 + de], 1);
  int cls = it_armor(type) ? 0 : it_weapon(type) ? 1 : it_tool(type) ? 2 : it_ammo(type) ? 3 : it_consumable(type) ? 4 : -1;
  if (de == 9 && cls >= 0 && cls < 4) atomicOr(&st[ST_EQUIP_FLAGS], 1 << cls);
  if (de == 8 && cls == 1) atomicOr(&st[ST_EQUIP_FLAGS], 1 << 4);
  if (de == 2) atomicMax(&st[ST_MAX_PROGRESS], number);
  if (de == 13) atomicAdd(&st[ST_EARNED_GOLD], gold);
  if (de == 3) atomicMax(&st[ST_MAX_DAMAGE], number);
  if ((de == 8 || de == 10 || de == 14) && cls >= 0) atomicMax(&st[ST_MAXLVL_ARMOR + cls], level);
  if (de == 4) { if (tpos) atomicAdd(&st[ST_AGENT_KILLS], 1); else if (tneg) atomicAdd(&st[ST_NPC_KILLS], 1); }
  // unique (event, type, level)
  int bit = (de * IT_N + type) * NM_UNIQ_LEVELS + min(level, NM_UNIQ_LEVELS - 1);
  uint32_t m = 1u << (bit & 31);
  uint32_t old = atomicOr(&ctx.p->uniq[a * NM_UNIQ_WORDS + (bit >> 5)], m);
  if (!(old & m) || de == 4 || de == 13) atomicAdd(&ctx.duniq[agent], 1);
  // event-driven predicate accumulators
  int pred = ctx.task[agent * 4], p0 = ctx.task[agent * 4 + 1], p1 = ctx.task[agent * 4 + 2];
  int *acc = ctx.acc + agent * 2;
  switch (pred) {
    case TP_COUNT_EVENT: if (nm_dense_event(p0) == de) atomicAdd(&acc[0], 1); break;
    case TP_SCORE_HIT: if (de == 3 && type == p0) atomicAdd(&acc[0], 1); break;
    case TP_EARN_GOLD: if (de == 13) atomicAdd(&acc[0], gold); break;
    case TP_SPEND_GOLD: if (de == 14) atomicAdd(&acc[0], gold); break;
    case TP_MAKE_PROFIT: if (de == 13) atomicAdd(&acc[0], gold); if (de == 14) atomicAdd(&acc[1], gold); break;
    case TP_CONSUME_ITEM: if (de == 5 && type == p0 && level >= p1) atomicAdd(&acc[0], number); break;
    case TP_HARVEST_ITEM: if (de == 8 && type == p0 && level >= p1) atomicAdd(&acc[0], number); break;
    case TP_LIST_ITEM: if (de == 12 && type == p0 && level >= p1) atomicAdd(&acc[0], number); break;
    case TP_BUY_ITEM: if (de == 14 && type == p0 && level >= p1) atomicAdd(&acc[0], number); break;
    case TP_DEFEAT_ENTITY: if (de == 4 && (p0 ? tpos : tneg) && level >= p1) atomicAdd(&acc[0], 1); break;
    default: break;
  }
}

// episode-end info record (stat_wrapper.py:132-185, :216-288)
template <class V>
__device__ void write_info(const Ctx<V> &ctx, int p, bool terminated, double cum_reward, double max_progress,
                           int reward_signals, int completed, int unique_events) {
  size_t a = (size_t)ctx.env * ctx.P + p;
  float *o = ctx.p->info + a * IN_N;
  const int32_t *st = ctx.p->stats + a * ST_N;
  float v[IN_N];
#pragma unroll
  for (int i = 0; i < IN_N; i++) v[i] = 0.0f;
  v[IN_LENGTH] = (float)ctx.tick;
  v[IN_RETURN] = (float)cum_reward;
  if (terminated) {
    v[IN_COD_ATTACKED] = ENT(EA_DAMAGE, p) > 0 ? 1.0f : 0.0f;
    v[IN_COD_STARVED] = ENT(EA_FOOD, p) == 0 ? 1.0f : 0.0f;
    v[IN_COD_DEHYDRATED] = ENT(EA_WATER, p) == 0 ? 1.0f : 0.0f;
  }
  v[IN_TASK_COMPLETED] = completed ? 1.0f : 0.0f;
  v[IN_TASK_2_REWARD_SIGNAL] = reward_signals >= 2 ? 1.0f : 0.0f;
  v[IN_TASK_0P2_MAX_PROGRESS] = max_progress >= 0.2 ? 1.0f : 0.0f;
  v[IN_CURR_MAX_PROGRESS] = (float)max_progress;
  v[IN_CURR_REWARD_SIGNALS] = (float)reward_signals;
  if (ctx.c[NC_EVAL_MODE]) v[IN_RETURN] = (float)max_progress;
  v[IN_MAX_COMBAT_LEVEL] = (float)attack_level(ctx, p);
  v[IN_MAX_HARVEST_AMMO] = (float)max((int)ENT(EA_PROSPECTING_LEVEL, p), max((int)ENT(EA_CARVING_LEVEL, p), (int)ENT(EA_ALCHEMY_LEVEL, p)));
  v[IN_MAX_HARVEST_CONSUM] = (float)max((int)ENT(EA_FISHING_LEVEL, p), (int)ENT(EA_HERBALISM_LEVEL, p));
  v[IN_MAX_PROGRESS_TO_CENTER] = (float)__ldcg(&st[ST_MAX_PROGRESS]);
  v[IN_EARNED_GOLD] = (float)__ldcg(&st[ST_EARNED_GOLD]);
  v[IN_MAX_DAMAGE] = (float)__ldcg(&st[ST_MAX_DAMAGE]);
  for (int k = 0; k < 5; k++) { int l = __ldcg(&st[ST_MAXLVL_ARMOR + k]); v[IN_MAXLVL_ARMOR + k] = l >= 0 ? (float)l : __int_as_float(0x7fc00000); }
  v[IN_AGENT_KILLS] = (float)__ldcg(&st[ST_AGENT_KILLS]);
  v[IN_NPC_KILLS] = (float)__ldcg(&st[ST_NPC_KILLS]);
  v[IN_UNIQUE_EVENTS] = (float)unique_events;
  v[IN_EV_EAT_FOOD] = __ldcg(&st[ST_EVT0 + 0]) > 0; v[IN_EV_DRINK_WATER] = __ldcg(&st[ST_EVT0 + 1]) > 0;
  v[IN_EV_SCORE_HIT] = __ldcg(&st[ST_EVT0 + 3]) > 0; v[IN_EV_PLAYER_KILL] = __ldcg(&st[ST_EVT0 + 4]) > 0;
  v[IN_EV_CONSUME_ITEM] = __ldcg(&st[ST_EVT0 + 5]) > 0; v[IN_EV_HARVEST_ITEM] = __ldcg(&st[ST_EVT0 + 8]) > 0;
  v[IN_EV_LIST_ITEM] = __ldcg(&st[ST_EVT0 + 12]) > 0; v[IN_EV_BUY_ITEM] = __ldcg(&st[ST_EVT0 + 14]) > 0;
  int fl = __ldcg(&st[ST_EQUIP_FLAGS]);
  for (int k = 0; k < 4; k++) v[IN_EQUIP_ARMOR + k] = (float)((fl >> k) & 1);
  v[IN_HARVEST_WEAPON] = (float)((fl >> 4) & 1);
  v[IN_TASK_ID] = (float)ctx.p->task_id[a];
  // running sums for nmmo_stats(): NM_AGG_REP replicas (picked by env) keep thousands of agents
  // that finish in the same tick from queueing on 80 addresses; zero terms are skipped, and the
  // count of a key that cannot be NaN is the count of finished agents (slot 0)
  double *ag = ctx.p->agg + (size_t)(ctx.env & (NM_AGG_REP - 1)) * (2 * IN_N);
#pragma unroll
  for (int i = 0; i < IN_N; i += 4) *(float4 *)(o + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
#pragma unroll
  for (int i = 0; i < IN_N; i++) {
    if (v[i] == v[i] && v[i] != 0.0f) atomicAdd(&ag[i], (double)v[i]);
    if (i >= IN_MAXLVL_ARMOR && i <= IN_MAXLVL_CONSUMABLE && v[i] == v[i]) atomicAdd(&ag[IN_N + i], 1.0);
  }
  atomicAdd(&ag[IN_N], 1.0);
  ctx.p->info_valid[a] = 1;
}

// ------------------------------------------------------------------------ reset -----
#ifndef NM_RESET_INLINE
#define NM_RESET_INLINE __noinline__
#endif
template <class V>
__device__ NM_RESET_INLINE void reset_env(const NmParams &P_, int env, uint64_t seed, bool explicit_map, bool explicit_tasks,
                          int *s_slot /* >= 2*P ints of shared memory */) {
  const int32_t *c = P_.cfg;
  int tid = threadIdx.x % V::kThreads, T = V::kThreads;
  const int half_id = threadIdx.x / V::kThreads;
  int P = P_.P, R = P_.R, S = P_.S;
  int32_t *sc = P_.scalars + (size_t)env * NM_SC_N;
  // injected draws are keyed by tick 0 here
  Ctx<V> ctx;
  ctx.p = &P_; ctx.c = NmCfg<V::kStd>{c}; ctx.env = env; ctx.seed = seed; ctx.tick = 0;
  ctx.inj_lo = P_.inj_off ? P_.inj_off[env] : 0; ctx.inj_hi = P_.inj_off ? P_.inj_off[env + 1] : 0;
  int map_id = explicit_map ? sc[SC_MAP_ID] : nm_bounded(draw(ctx, RS_MAP, 0, 0), P_.n_maps);
  // map copy, table clears
  {
    // source maps are one byte per tile; the live map packs two tiles per byte
    const uint2 *src = (const uint2 *)(P_.maps + (size_t)map_id * S * S);
    uint32_t *dst = (uint32_t *)(P_.map + (size_t)env * (S * S / 2));
    #pragma unroll 1
    for (int i = tid; i < S * S / 8; i += T) {
      uint2 b = src[i];
      uint32_t lo = b.x, hi = b.y;
      dst[i] = (lo & 15u) | ((lo >> 4) & 0xf0u) | ((lo >> 8) & 0xf00u) | ((lo >> 12) & 0xf000u) |
               ((hi & 15u) << 16) | (((hi >> 8) & 15u) << 20) | (((hi >> 16) & 15u) << 24) | (((hi >> 24) & 15u) << 28);
    }
    uint4 z = make_uint4(0, 0, 0, 0);
    const size_t ent_i16 = V::kGlobalTables ? (size_t)NM_BIG_ENT_STRIDE * R : (size_t)EA_N * R;      // int16 per env
    uint4 *e4 = (uint4 *)(P_.ent + (size_t)env * ent_i16);
    #pragma unroll 1
    for (int i = tid; i < (int)(ent_i16 * 2 / 16); i += T) e4[i] = z;
    // the item table is not cleared: SC_ITEM_HI = 0 below declares every row free
    uint32_t *u = P_.uniq + (size_t)env * P * NM_UNIQ_WORDS;
    #pragma unroll 1
    for (int i = tid; i < P * NM_UNIQ_WORDS; i += T) u[i] = 0;
    int32_t *st = P_.stats + (size_t)env * P * ST_N;
    #pragma unroll 1
    for (int i = tid; i < P * ST_N; i += T) { int k = i % ST_N; st[i] = (k >= ST_MAXLVL_ARMOR && k <= ST_MAXLVL_CONSUMABLE) ? -1 : (k == ST_Y_HP ? 100 : 0); }
    double *ds = P_.dstats + (size_t)env * P * DS_N;
    #pragma unroll 1
    for (int i = tid; i < P * DS_N; i += T) ds[i] = 0.0;
  }
  int *slot = s_slot, *resil = s_slot + P;
  if (tid == 0) {
    for (int i = 0; i < P; i++) { slot[i] = i; resil[i] = i < c[NC_RES_RESILIENT_N] ? 1 : 0; }
    for (int i = P - 1; i >= 1; i--) {
      int j = nm_bounded(draw(ctx, RS_SPAWN_PERM, (uint32_t)i, 0), i + 1);
      int t = slot[i]; slot[i] = slot[j]; slot[j] = t;
    }
    for (int i = P - 1; i >= 1; i--) {
      int j = nm_bounded(draw(ctx, RS_RESILIENT, (uint32_t)i, 0), i + 1);
      int t = resil[i]; resil[i] = resil[j]; resil[j] = t;
    }
  }
  // barrier over this environment's own 256 threads (the other half of the CTA may be stepping, or gone)
  asm volatile("bar.sync %0, %1;" ::"r"(1 + half_id), "r"(V::kThreads) : "memory");      // also orders the table clears before the row writes below
  int16_t *ent = P_.ent + (size_t)env * (V::kGlobalTables ? (size_t)NM_BIG_ENT_STRIDE * R : (size_t)EA_N * R);
  const int patch = c[NC_SPAWN_PATCH];
  int b = c[NC_MAP_BORDER], ce = c[NC_MAP_CENTER];
  #pragma unroll 1
  for (int p = tid; p < P; p += T) {
    int k = (int)(((long long)slot[p] * (4 * ce)) / P);
    int side = k / ce, off = k % ce, r, cc;
    if (side == 0) { r = b; cc = b + off; }
    else if (side == 1) { r = b + off; cc = b + ce; }
    else if (side == 2) { r = b + ce; cc = b + ce - off; }
    else { r = b + ce - off; cc = b; }
    if (patch > 0) {      // stress workload (BASELINE.json configs[4]): shuffled cells of a patch x patch square at the centre
      const int o = S / 2 - patch / 2, cell = (int)(((long long)slot[p] * patch * patch) / P);
      r = o + cell / patch; cc = o + cell % patch;
    }
#define GENT(col) ent[V::ent_idx((col), p, R)]
    GENT(EA_ID) = (int16_t)(p + 1); GENT(EA_ROW) = (int16_t)r; GENT(EA_COL) = (int16_t)cc;
    GENT(EA_GOLD) = (int16_t)c[NC_BASE_GOLD]; GENT(EA_HEALTH) = (int16_t)c[NC_RES_BASE];
    GENT(EA_FOOD) = (int16_t)c[NC_RES_BASE]; GENT(EA_WATER) = (int16_t)c[NC_RES_BASE];
    for (int col = EA_MELEE_LEVEL; col <= EA_ALCHEMY_LEVEL; col += 2) GENT(col) = 1;
    GENT(EA_SPAWN_ROW) = (int16_t)r; GENT(EA_SPAWN_COL) = (int16_t)cc; GENT(EA_RESILIENT) = (int16_t)resil[p];
    GENT(EA_STATUS) = ES_ALIVE;
#undef GENT
    size_t a = (size_t)env * P + p;
    // one task per team: the draw is keyed by the team leader's row (team size 1: by the agent's own)
    if (!explicit_tasks) P_.task_id[a] = nm_bounded(draw(ctx, RS_TASK, (uint32_t)(p - p % max(1, c[NC_TEAM_SIZE])), 0), P_.n_tasks);
    P_.rew[a] = 0.0f; P_.term[a] = 0; P_.trunc[a] = 0; P_.mask[a] = 1; P_.info_valid[a] = 0;
    P_.obs_meta[a] &= ~OM_TASK;        // new episode, new task embedding
  }
  if (tid == 0) {
    P_.seed[env] = seed;
    sc[SC_TICK] = 0; sc[SC_DONE] = 0; sc[SC_NEXT_NPC_ID] = -1; sc[SC_N_DANGER] = 0; sc[SC_MAP_ID] = map_id;
    sc[SC_FRESH] = 1; sc[SC_ITEM_HI] = 0; sc[SC_N_DEPL] = 0; sc[SC_NEED_RESET] = 0; sc[SC_EXPLICIT_MAP] = 0; sc[SC_EXPLICIT_TASKS] = 0;
    P_.episode_done[env] = 0;
    if (P_.ev_n) P_.ev_n[env] = 0;      // a reset env has no events in the event log
  }
}

}  // namespace

// Barriers over one environment's threads (named barrier 1 + half).  In the small family two environments share a
// CTA so that they walk the kernel's code together (one instruction fetch serves both); they never wait for each other.
#define HSYNC() asm volatile("bar.sync %0, %1;" ::"r"(1 + half), "n"(V::kThreads) : "memory")
template <int NT>
__device__ __forceinline__ int half_or_t(int pred, int half) {
  int r;
  asm volatile("{ .reg .pred p, q; setp.ne.s32 p, %1, 0; bar.red.or.pred q, %2, %3, p; selp.s32 %0, 1, 0, q; }"
               : "=r"(r) : "r"(pred), "r"(1 + half), "n"(NT) : "memory");
  return r;
}
template <int NT>
__device__ __forceinline__ int half_count_t(int pred, int half) {
  int r;
  asm volatile("{ .reg .pred p; setp.ne.s32 p, %1, 0; bar.red.popc.u32 %0, %2, %3, p; }"
               : "=r"(r) : "r"(pred), "r"(1 + half), "n"(NT) : "memory");
  return r;
}
#define half_or(pred, half) half_or_t<V::kThreads>((pred), (half))
#define half_count(pred, half) half_count_t<V::kThreads>((pred), (half))

// ===================================================================== step kernel ====
template <class V>
__device__ __forceinline__ void step_body(const NmParams &prm) {
  // Small family: two environments per CTA, 256 threads and half of the dynamic shared memory each.  They share
  // nothing and never wait for each other (every barrier below is a named barrier over one half); the point of the
  // pairing is that both walk the kernel's 300 KB of code at the same time, so the SM fetches it once
  // (measured: 0.63 -> 0.56 ms against two independent 256-thread CTAs per SM, DESIGN.md 4.1).
  // Big family: one environment per CTA (half == 0).
  typedef typename V::tile_t tile_t;
  extern __shared__ __align__(128) uint8_t smem_all[];
  const int half = threadIdx.x / V::kThreads;
  uint8_t *smem = smem_all + (size_t)half * prm.half_smem;
  const int env = prm.env_lo + blockIdx.x * prm.envs_per_cta + half, tid = threadIdx.x % V::kThreads, T = V::kThreads, lane = tid & 31, warp = tid >> 5;
  const NmCfg<V::kStd> c{prm.cfg};
  constexpr nm_obs_layout kStdL = nm_std_layout();
  typedef typename V::Shape SH;
  const int P = V::kStd ? SH::P : prm.P, N = V::kStd ? SH::N : prm.N, R = V::kStd ? SH::R : prm.R;
  const int S = V::kStd ? SH::S : prm.S, CAP = V::kStd ? SH::CAP : prm.CAP, NINV = V::kStd ? SH::NINV : c[NC_N_INV];
  if (env >= prm.env_hi) return;     // odd environment count: the last CTA runs one half (exited threads do not count at barriers)
  int32_t *gsc = prm.scalars + (size_t)env * NM_SC_N;

  // ---- reset paths -------------------------------------------------------------------
  if (prm.mode == 1) {
    if (!gsc[SC_NEED_RESET]) return;
    reset_env<V>(prm, env, prm.seed[env], gsc[SC_EXPLICIT_MAP] != 0, gsc[SC_EXPLICIT_TASKS] != 0, (int *)smem);
    return;
  }

  // ---- shared memory carve-up ---------------------------------------------------------
  size_t off = 0, goff = 0;
  auto carve = [&](size_t bytes) { uint8_t *q = smem + off; off = (off + bytes + 15) & ~(size_t)15; return q; };
  // big family: the arrays that are touched a few times per tick live in a per-env workspace in HBM / L2
  uint8_t *const gws = V::kItemsInPlace ? prm.ws + (size_t)env * prm.ws_bytes : nullptr;
  // in_ws: the array goes to the workspace (big family and VSmall4: act / task / acc; VSmall4 only: the rest)
  auto carve_ws = [&](size_t bytes, bool in_ws = V::kGlobalTables || V::kScratchInWs) {
    if (!in_ws) return carve(bytes);
    uint8_t *q = gws + goff; goff = (goff + bytes + 15) & ~(size_t)15; return q;
  };
  const uint32_t ent_bytes = (uint32_t)(EA_N * R * 2), item_bytes = (uint32_t)(IS_N * CAP * 2), map_bytes = (uint32_t)(S * S / 2);
  Ctx<V> ctx;
  ctx.p = &prm; ctx.c = c; ctx.env = env; ctx.P = P; ctx.N = N; ctx.R = R; ctx.S = S; ctx.CAP = CAP; ctx.NINV = NINV;
  int16_t *const gitem = prm.item + (size_t)env * IS_N * CAP;
  if (V::kGlobalTables) {
    ctx.ent = prm.ent + (size_t)env * NM_BIG_ENT_STRIDE * R;
    ctx.item = gitem;
    ctx.map = (uint32_t *)(prm.map + (size_t)env * map_bytes);
  } else {
    ctx.ent = (int16_t *)carve(ent_bytes);
    ctx.item = V::kItemsInPlace ? gitem : (int16_t *)carve(item_bytes);
    ctx.map = (uint32_t *)carve(map_bytes);
  }
  const int occ_words = (S * S + 31) >> 5, cap_words = (CAP + 31) >> 5;
  ctx.occ = (uint32_t *)carve(occ_words * 4);
  ctx.used = (uint32_t *)carve(cap_words * 4);
  ctx.fresh = (uint32_t *)carve(cap_words * 4);
  ctx.inv = (uint16_t *)carve_ws((size_t)P * NINV * 2, V::kScratchInWs);
  ctx.invn = carve(P);
  ctx.act = (int16_t *)carve_ws((size_t)A_N * P * 2);
  ctx.npc_move = (int8_t *)carve(N);
  ctx.npc_att = (int16_t *)carve((size_t)N * 2);
  if (V::kItemsInPlace && !V::kGlobalTables) { ctx.ev = (uint2 *)(gws + goff); goff += (size_t)V::kEvCap * 8; }      // (VSmall3: the only workspace array)
  else ctx.ev = (uint2 *)carve_ws((size_t)V::kEvCap * 8);
  ctx.duniq = (int *)carve_ws((size_t)P * 4, V::kScratchInWs);
  int *s_list = V::kScratchInWs ? nullptr : (int *)carve((size_t)P * 4);      // (VSmall4: in the scratch, below)
  ctx.npc_hash = (unsigned short *)carve((size_t)V::kNpcHash * 2);
  ctx.task = (int *)carve_ws((size_t)P * 16);
  ctx.acc = (int *)carve_ws((size_t)P * 8);
  // 4 KB scratch reused phase by phase: attack list + registrations, move tile hash,
  // respawn worklist, NPC-spawn pre-drawn values
  const size_t scratch_bytes = max((size_t)4096, (size_t)R * 8);
  // + the per-chunk counts behind the two attack arrays (VSmall4: R <= 384, they fit in the 4 KB)
  uint32_t *s_scratch = (uint32_t *)carve(scratch_bytes + (V::kScratchInWs ? 0 : 32 * V::kChunkIters * 4));
  uint8_t *s_mv = carve((size_t)R * (sizeof(tile_t) + 2));     // Move phase: destination (tile_t) + verdict (u16) per row; >= R * 4 bytes
  // depleted-tile list: staged in shared memory (small) / used in place in HBM (big, VSmall4)
  constexpr bool kDeplInPlace = V::kGlobalTables || V::kScratchInWs;
  tile_t *const gdepl = (tile_t *)prm.depl + (size_t)env * V::kDeplCap;
  ctx.dlist = kDeplInPlace ? gdepl : (tile_t *)carve((size_t)V::kDeplCap * sizeof(tile_t));
  // Move phase: position index (tile -> row).  VSmall4: in the scratch, which the attack phase leaves before the Move
  uint32_t *s_tbl = V::kScratchInWs ? s_scratch : (uint32_t *)carve((size_t)V::kTblSlots * 4);
  static_assert(!V::kScratchInWs || V::kTblSlots * 4 <= 4096, "the position index must fit the scratch");
  // VSmall4: the player list of the update / harvest / Buy phases and of the window scans sits in the scratch behind
  // the first 2 KB (idle in those phases; the depleted-tile list the writeback copies out of it is <= 2 KB)
  if (V::kScratchInWs) s_list = (int *)(s_scratch + 512);
  static_assert(!V::kScratchInWs || (V::kThreads + 512) * 4 <= 4096, "the player list must fit the scratch");
  uint32_t *s_att = s_scratch;
  int *s_first = (int *)(s_scratch + R);
  ctx.slow = (int8_t *)carve_ws((size_t)P, V::kScratchInWs);
  // alive players for the NPC target scans (phases 0-1).  VSmall4: in the Move scratch, which the attack phase is first to use
  uint32_t *s_plist = V::kScratchInWs ? (uint32_t *)s_mv : (uint32_t *)carve((size_t)P * 4);
  ctx.sc = (int *)carve(32 * 4);
  uint64_t *bar = (uint64_t *)carve(16);
  // ---- load: three bulk copies on one mbarrier, issued before anything else touches HBM ----
  if (!V::kGlobalTables) {
  if (tid == 0) {
    mbar_init(bar, 1); mbar_init(bar + 1, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  HSYNC();
  if (tid == 0) {
    mbar_expect_tx(bar, ent_bytes + map_bytes);
    bulk_g2s(ctx.ent, prm.ent + (size_t)env * EA_N * R, ent_bytes, bar);
    bulk_g2s(ctx.map, prm.map + (size_t)env * map_bytes, map_bytes, bar);
  }
  }
  const int done_flag = gsc[SC_DONE];      // consumed below, after the other loads are in flight
  const int item_hi0 = gsc[SC_ITEM_HI];    // rows >= item_hi0 are free (multiple of 8)
  const int n_depl0 = gsc[SC_N_DEPL];      // depleted tiles listed in prm.depl (-1: list unknown)
  if (!V::kGlobalTables && tid == 0) {
    // Item rows are allocated lowest-free-first, so live rows crowd the low end of the table: only
    // the prefix below the high-water mark moves between HBM and shared memory.  Rows above it are
    // never read before they are allocated (the in-use bitmap is built from the prefix).
    const uint32_t col_bytes = (uint32_t)item_hi0 * 2;
    const uint32_t dl_bytes = n_depl0 > 0 && !kDeplInPlace ? (uint32_t)((n_depl0 * (int)sizeof(tile_t) + 15) & ~15) : 0u;
    mbar_expect_tx(bar + 1, (V::kItemsInPlace ? 0u : col_bytes * IS_N) + dl_bytes);
    if (dl_bytes) bulk_g2s(ctx.dlist, gdepl, dl_bytes, bar + 1);
    if (col_bytes && !V::kItemsInPlace)
      for (int k = 0; k < IS_N; k++) bulk_g2s(ctx.item + k * CAP, gitem + (size_t)k * CAP, col_bytes, bar + 1);
  }
  ctx.seed = prm.seed[env];
  ctx.tick = gsc[SC_TICK];
  ctx.inj_lo = prm.inj_off ? prm.inj_off[env] : 0;
  ctx.inj_hi = prm.inj_off ? prm.inj_off[env + 1] : 0;

  // per-player wrapper state: issued now, consumed at the end of the step
  const size_t my_a = (size_t)env * P + (tid < P ? tid : 0);
  int32_t *my_sta = prm.stats + my_a * ST_N;
  double *my_ds = prm.dstats + my_a * DS_N;
  int my_task_id = 0, my_t[NM_TASK_COLS] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};
  int my_done = 0, my_signals = 0, my_uniq = 0, my_acc0 = 0, my_acc1 = 0;
  double my_cum = 0.0, my_prog = 0.0, my_maxprog = 0.0;
  if (tid < P) {
    my_task_id = prm.task_id[my_a];
    const int4 *tr = (const int4 *)(prm.tasks + (size_t)my_task_id * NM_TASK_COLS);
    int4 t0 = __ldg(tr), t1 = __ldg(tr + 1), t2 = __ldg(tr + 2);
    my_t[8] = t2.x; my_t[9] = t2.y; my_t[10] = t2.z; my_t[11] = t2.w;
    my_t[0] = t0.x; my_t[1] = t0.y; my_t[2] = t0.z; my_t[3] = t0.w; my_t[4] = t1.x; my_t[5] = t1.y; my_t[6] = t1.z; my_t[7] = t1.w;
    my_done = my_sta[ST_TASK_DONE]; my_signals = my_sta[ST_REWARD_SIGNALS]; my_uniq = my_sta[ST_UNIQ_CURR];
    my_acc0 = my_sta[ST_TASK_ACC0]; my_acc1 = my_sta[ST_TASK_ACC1];
    my_cum = my_ds[DS_CUM_REWARD]; my_prog = my_ds[DS_PROGRESS]; my_maxprog = my_ds[DS_MAX_PROGRESS];
  }
  long long t_prev = clock64();
  int ph = 0;
  // (the *_std instantiations carry neither the per-phase profile counters nor the injected-draw lookup: a handle that
  //  profiles or injects draws launches the generic instantiation)
#define PHASE() do { if (!V::kStd && prm.prof && tid == 0) { long long t_ = clock64(); atomicAdd(&prm.prof[ph], (unsigned long long)(t_ - t_prev)); t_prev = t_; } ph++; } while (0)
#define PCOUNT(slot, v) do { if (!V::kStd && prm.prof && tid == 0) atomicAdd(&prm.prof[slot], (unsigned long long)(v)); } while (0)
  #pragma unroll 1
  for (int i = tid; i < occ_words; i += T) ctx.occ[i] = 0;
  #pragma unroll 1
  for (int i = tid; i < cap_words; i += T) { ctx.used[i] = 0; ctx.fresh[i] = 0; }
  #pragma unroll 1
  for (int i = tid; i < P; i += T) { ctx.invn[i] = 0; ctx.duniq[i] = 0; }
  #pragma unroll 1
  for (int i = tid; i < V::kNpcHash / 2; i += T) ((uint32_t *)ctx.npc_hash)[i] = 0;
  #pragma unroll 1
  for (int i = tid; i < (V::kScratchInWs ? 0 : V::kTblSlots); i += T) s_tbl[i] = 0;
  if (tid < P) {
    ctx.task[tid * 4] = my_t[0]; ctx.task[tid * 4 + 1] = my_t[1]; ctx.task[tid * 4 + 2] = my_t[2]; ctx.task[tid * 4 + 3] = 0;
    ctx.acc[tid * 2] = my_acc0; ctx.acc[tid * 2 + 1] = my_acc1;
  }
  if (tid < 32) ctx.sc[tid] = 0;
  if (tid == 0) { ctx.sc[2] = gsc[SC_N_DANGER]; ctx.sc[3] = gsc[SC_NEXT_NPC_ID]; ctx.sc[17] = max(n_depl0, 0); }
  if (done_flag) {      // episode over: this launch resets the environment instead of stepping it
    if (!V::kGlobalTables) {
      while (!mbar_try_wait(bar, 0)) {}      // the bulk copies must have landed before shared memory is reused
      while (!mbar_try_wait(bar + 1, 0)) {}
    }
    HSYNC();
    if (tid == 0) { gsc[SC_EPISODE] += 1; atomicAdd(&prm.counters[2], 1ULL); }
    reset_env<V>(prm, env, nm_mix64(ctx.seed + 0x632BE59BD9B4E019ULL), false, false, (int *)smem);
    return;
  }
  // Decode the player actions against the observation record they were chosen on (the ids are read
  // back from the record in HBM).  Only global memory is involved, so these loads overlap the bulk
  // copies; targets stay entity ids here and become table rows once the tables have landed.
  int my_prev_price = 0;
  if (tid < P) {
    const int p = tid;
    const int4 *x4 = (const int4 *)(prm.actions + ((size_t)(env - prm.act_env_lo) * P + p) * AC_N);
    const int16_t *gent = prm.ent + (size_t)env * (V::kGlobalTables ? (size_t)NM_BIG_ENT_STRIDE * R : (size_t)EA_N * R);
    const int g_status = gent[V::ent_idx(EA_STATUS, p, R)], g_health = gent[V::ent_idx(EA_HEALTH, p, R)];   // same answer as ent_alive() later
    int4 xa = x4[0], xb = x4[1], xc = x4[2];
    if (!(g_status == ES_ALIVE && g_health > 0)) { xa = make_int4(-1, -1, -1, -1); xb = xa; xc = xa; }   // no id reads for the dead
    const nm_obs_layout &L = V::kStd ? kStdL : prm.L;
    const uint8_t *rec = prm.obs + ((size_t)env * P + p) * L.stride;
    auto ent_id = [&](int idx) -> int { return (idx >= 0 && idx < L.n_ent) ? (int)*(const int16_t *)(rec + L.o_entity + idx * (EA_N_OBS * 2)) : 0; };
    auto inv_id = [&](int idx) -> int { return (idx >= 0 && idx < L.n_inv) ? (int)*(const int16_t *)(rec + L.o_inventory + idx * (IA_N_OBS * 2)) : 0; };
    auto mkt_id = [&](int idx) -> int { return (idx >= 0 && idx < L.n_mkt) ? (int)*(const int16_t *)(rec + L.o_market + idx * (IA_N_OBS * 2)) : 0; };
    const int a_as = xa.x, a_at = xa.y, a_buy = xa.z, a_des = xa.w, a_gi = xb.x, a_gt = xb.y, a_gp = xb.z, a_gg = xb.w;
    const int a_mv = xc.x, a_si = xc.y, a_sp = xc.z, a_use = xc.w;
    // all eight id reads are independent: issue them together
    const int i_use = inv_id(a_use), i_des = inv_id(a_des), i_si = inv_id(a_si), i_buy = mkt_id(a_buy), i_gi = inv_id(a_gi);
    const int t_gt = ent_id(a_gt), t_gg = ent_id(a_gg), t_at = ent_id(a_at);
    int16_t v[A_N];
#pragma unroll
    for (int k = 0; k < A_N; k++) v[k] = 0;
    v[A_MOVE] = -1;
    v[A_USE] = (int16_t)i_use;
    v[A_DESTROY] = (int16_t)i_des;
    const bool sp_ok = a_sp >= 0 && a_sp < L.n_price;
    if (sp_ok && i_si) { v[A_SELL_ITEM] = (int16_t)i_si; v[A_SELL_PRICE] = (int16_t)(a_sp + 1); }
    v[A_BUY] = (int16_t)i_buy;
    if (i_gi && t_gt > 0) { v[A_GIVE_ITEM] = (int16_t)i_gi; v[A_GIVE_TARGET] = (int16_t)t_gt; }
    if (a_gp >= 0 && a_gp < L.n_price && t_gg > 0) { v[A_GOLD_AMT] = (int16_t)(a_gp + 1); v[A_GOLD_TARGET] = (int16_t)t_gg; }
    if (a_as >= 0 && a_as < 3 && t_at) { v[A_ATT_STYLE] = (int16_t)a_as; v[A_ATT_TARGET] = (int16_t)t_at; }
    if (a_mv >= 0 && a_mv < 4) v[A_MOVE] = (int16_t)a_mv;
    my_prev_price = sp_ok ? a_sp : 0;
#pragma unroll
    for (int k = 0; k < A_N; k++) ctx.act[k * P + p] = v[k];
  }
  if (!V::kGlobalTables) {
    while (!mbar_try_wait(bar, 0)) {}
    while (!mbar_try_wait(bar + 1, 0)) {}
  }
  HSYNC();

  PHASE();
  // ---- phase 0: bookkeeping rebuilt from the tables -----------------------------------
  // one pass over the rows: last tick's dead players become empty slots, alive entities enter the occupancy bitmap,
  // alive NPCs the id -> row hash (read by the validation below, after the barrier)
  #pragma unroll 1
  for (int r = tid; r < R; r += T) {
    const int st = ENT(EA_STATUS, r);
    if (st == ES_DEAD_THIS_TICK && r < P) ENT(EA_STATUS, r) = ES_EMPTY;
    if (st == ES_ALIVE) {
      occ_set(ctx, ENT(EA_ROW, r), ENT(EA_COL, r));
      if (r >= P) {
        unsigned h = (((unsigned)(-(int)ENT(EA_ID, r))) * 40503u >> 4) & (unsigned)(V::kNpcHash - 1);
        #pragma unroll 1
        while (atomicCAS(&ctx.npc_hash[h], (unsigned short)0, (unsigned short)(r + 1)) != 0) h = (h + 1) & (unsigned)(V::kNpcHash - 1);
      }
    }
  }
  if (warp == 0) {       // alive players, ascending id, with packed positions (NPC target scans)
    int n = 0;
    #pragma unroll 1
    for (int base = 0; base < P; base += 32) {
      int p = base + lane;
      bool live = p < P && ENT(EA_STATUS, p) == ES_ALIVE;
      unsigned bm = __ballot_sync(0xffffffffu, live);
      if (live) s_plist[n + __popc(bm & ((1u << lane) - 1))] = ((uint32_t)p << 20) | ((uint32_t)ENT(EA_ROW, p) << 10) | (uint32_t)ENT(EA_COL, p);
      n += __popc(bm);
    }
    if (lane == 0) ctx.sc[16] = n;
  }
  #pragma unroll 1
  for (int g = tid; g < item_hi0 / 8; g += T) {      // 8 rows of the type column per 16-byte load
    const uint4 t8 = ((const uint4 *)(ctx.item + IS_TYPE * CAP))[g];
    if (!(t8.x | t8.y | t8.z | t8.w)) continue;
    const uint32_t tw[4] = {t8.x, t8.y, t8.z, t8.w};
#pragma unroll
    for (int j = 0; j < 8; j++) {
      if (!((tw[j >> 1] >> ((j & 1) * 16)) & 0xffffu)) continue;
      const int i = g * 8 + j;
      atomicOr(&ctx.used[i >> 5], 1u << (i & 31));
      int owner = ITM(IS_OWNER, i);
      if (owner > 0) {
        // per-owner list; slot order is irrelevant to the engine (obs re-sorts by row)
        unsigned int *w = (unsigned int *)(ctx.invn + ((owner - 1) & ~3));
        int sh = ((owner - 1) & 3) * 8;
        unsigned int old = atomicAdd(w, 1u << sh);
        int slot = (old >> sh) & 255;
        ctx.inv[(owner - 1) * NINV + slot] = (uint16_t)i;
      }
    }
  }
  HSYNC();
  // ---- validate: entity ids chosen from the observation -> table rows; dead agents act on nothing
  if (tid < P) {
    const int p = tid;
    if (ent_alive(ctx, p)) {
      auto ent_row1 = [&](int id) -> int {
        if (id > 0) return id <= P ? id : 0;
        if (id < 0) {
          unsigned h = (((unsigned)(-id)) * 40503u >> 4) & (unsigned)(V::kNpcHash - 1);
          #pragma unroll 1
          for (int probe = 0; probe < V::kNpcHash; probe++) {
            int r1 = ctx.npc_hash[h];
            if (r1 == 0) return 0;
            if (ENT(EA_ID, r1 - 1) == id) return r1;
            h = (h + 1) & (unsigned)(V::kNpcHash - 1);
          }
        }
        return 0;
      };
      if (ctx.act[A_GIVE_ITEM * P + p]) ctx.act[A_GIVE_TARGET * P + p] = (int16_t)ent_row1(ctx.act[A_GIVE_TARGET * P + p]);
      if (ctx.act[A_GOLD_AMT * P + p]) ctx.act[A_GOLD_TARGET * P + p] = (int16_t)ent_row1(ctx.act[A_GOLD_TARGET * P + p]);
      if (ctx.act[A_ATT_TARGET * P + p]) ctx.act[A_ATT_TARGET * P + p] = (int16_t)ent_row1(ctx.act[A_ATT_TARGET * P + p]);
      if (c[NC_WRAPPER] == NW_START_KIT) prm.stats[((size_t)env * P + p) * ST_N + ST_PREV_PRICE] = my_prev_price;
    } else {
#pragma unroll
      for (int k = 0; k < A_N; k++) ctx.act[k * P + p] = k == A_MOVE ? (int16_t)-1 : (int16_t)0;
    }
  }
  {   // which item-action phases have anything to do this tick: the others are skipped together with their barriers
    int bits = 0;
    if (tid < P) {
      const int p = tid;
      bits = (ctx.act[A_USE * P + p] ? 1 : 0) | (ctx.act[A_BUY * P + p] ? 2 : 0) |
             ((ctx.act[A_GIVE_ITEM * P + p] || ctx.act[A_GOLD_AMT * P + p]) ? 4 : 0) | (ctx.act[A_DESTROY * P + p] ? 8 : 0) |
             (ctx.act[A_SELL_ITEM * P + p] ? 16 : 0);
    }
    bits = __reduce_or_sync(0xffffffffu, bits);
    if (lane == 0 && bits) atomicOr(&ctx.sc[23], bits);
  }
  HSYNC();

  PHASE();
  // ---- phase 1: npcs.actions ----------------------------------------------------------
  ctx.plist = s_plist; ctx.n_plist = ctx.sc[16];
  #pragma unroll 1
  for (int r = P + tid; r < R; r += T) {
    if (ent_alive(ctx, r)) npc_decide(ctx, r);
    else { ctx.npc_move[r - P] = -1; ctx.npc_att[r - P] = 0; }
  }
  HSYNC();

  PHASE();
  // ---- phase 2: players.update (order-free part), npcs.update -------------------------
  #pragma unroll 1
  for (int p = tid; p < P; p += T) {
    bool seq = false;
    if (ENT(EA_STATUS, p) == ES_ALIVE) {
      if (ENT(EA_DAMAGE, p) == 0) ENT(EA_ATTACKER_ID, p) = 0;
      int il = 0;
      #pragma unroll 1
      for (int s = EA_EQ_HAT; s <= EA_EQ_AMMO; s++) { int it = ENT(s, p); if (it) il += ITM(IS_LEVEL, it - 1); }
      ENT(EA_ITEM_LEVEL, p) = (int16_t)il;
      if (ENT(EA_FREEZE, p) > 0) ENT(EA_FREEZE, p) -= 1;
      ENT(EA_DAMAGE, p) = 0;
      ENT(EA_TIME_ALIVE, p) += 1;
      int hp = ENT(EA_HEALTH, p), org = hp, food = ENT(EA_FOOD, p), water = ENT(EA_WATER, p);
      if (food > c[NC_RES_REGEN_THRESH] && water > c[NC_RES_REGEN_THRESH]) hp = min(c[NC_RES_BASE], hp + c[NC_RES_HEALTH_RESTORE]);
      int res = ENT(EA_RESILIENT, p);
      if (food == 0) { int d = c[NC_RES_STARVATION]; if (res) d /= 2; hp = max(0, hp - d); }
      if (water == 0) { int d = c[NC_RES_DEHYDRATION]; if (res) d /= 2; hp = max(0, hp - d); }
      ENT(EA_HEALTH, p) = (int16_t)hp;
      ENT(EA_HEALTH_RESTORE, p) = (int16_t)(hp - org);
      int r = ENT(EA_ROW, p), cc = ENT(EA_COL, p);
      water = max(0, water - c[NC_RES_DEPLETION]);
      int up = tile_at(ctx, r - 1, cc), dn = tile_at(ctx, r + 1, cc), lf = tile_at(ctx, r, cc - 1), rt = tile_at(ctx, r, cc + 1);
      if (up == MT_WATER || dn == MT_WATER || lf == MT_WATER || rt == MT_WATER) {
        water = min(c[NC_RES_BASE], water + c[NC_RES_HARVEST_RESTORE]);
        emit(ctx, p, EV_DRINK_WATER, 0, 0, 0, 0, 0);
      }
      ENT(EA_WATER, p) = (int16_t)water;
      food = max(0, food - c[NC_RES_DEPLETION]);
      int here = tile_at(ctx, r, cc);
      if (here == MT_FOILAGE && !c[NC_ALLOW_OCCUPIED]) {
        // with one entity per tile nobody else can eat this tile: no ordering needed
        tile_dec(ctx, r * S + cc);
        food = min(c[NC_RES_BASE], food + c[NC_RES_HARVEST_RESTORE]);
        emit(ctx, p, EV_EAT_FOOD, 0, 0, 0, 0, 0);
        here = MT_SCRUB;
      }
      ENT(EA_FOOD, p) = (int16_t)food;
      seq = here == MT_FOILAGE || here == MT_HERB || here == MT_ORE || here == MT_TREE || here == MT_CRYSTAL ||
            up == MT_FISH || dn == MT_FISH || lf == MT_FISH || rt == MT_FISH;
    }
    s_list[p] = seq ? 1 : 0;
    if (seq) atomicOr(&ctx.sc[23], 32);
  }
  #pragma unroll 1
  for (int r = P + tid; r < R; r += T)
    if (ENT(EA_STATUS, r) == ES_ALIVE) {
      if (ENT(EA_DAMAGE, r) == 0) ENT(EA_ATTACKER_ID, r) = 0;
      if (ENT(EA_FREEZE, r) > 0) ENT(EA_FREEZE, r) -= 1;
      ENT(EA_DAMAGE, r) = 0;
      ENT(EA_TIME_ALIVE, r) += 1;
      if (ENT(EA_HEALTH, r) > 0) ENT(EA_HEALTH, r) = (int16_t)min(c[NC_RES_BASE], ENT(EA_HEALTH, r) + 1);
    }
  HSYNC();
  PHASE();
  const int todo = ctx.sc[23];      // env-uniform: bit per phase that has work (Use, Buy, Give, Destroy, Sell, harvest)
  // id-ordered part: tile depletion and drops
  if (todo & 32) {
  if (warp == 0) {
    #pragma unroll 1
    for (int base = 0; base < P; base += 32) {
      int p = base + lane;
      unsigned m = __ballot_sync(0xffffffffu, p < P && s_list[p]);
      #pragma unroll 1
      while (m) {
        int l = __ffs(m) - 1; m &= m - 1;
        if (lane == l) player_harvest(ctx, p);
        __syncwarp();
      }
    }
  }
  HSYNC();
  }

  PHASE();
  // ---- phase 3: actions in priority order ---------------------------------------------
  // Use (10): touches only the actor's own rows
  if (todo & 1) {
  #pragma unroll 1
  for (int p = tid; p < P; p += T) if (ent_alive(ctx, p) && ctx.act[A_USE * P + p]) act_use(ctx, p, ctx.act[A_USE * P + p]);
  HSYNC();
  }
  PHASE();
  // Buy (20): shuffled order.  Buyers are compacted in id order by the whole block, then
  // shuffled and executed by one thread (a handful per tick); Give / GiveGold (30) likewise
  if (todo & 6) {
    bool mine = tid < P && ctx.act[A_BUY * P + tid] && ent_alive(ctx, tid);
    unsigned bm = __ballot_sync(0xffffffffu, mine);
    int *const wcnt = V::kThreads > 256 ? (int *)s_scratch : &ctx.sc[8];      // per-warp buyer counts (the scratch is idle here)
    if (lane == 0) wcnt[warp] = __popc(bm);
    bool give = tid < P && (ctx.act[A_GIVE_ITEM * P + tid] || ctx.act[A_GOLD_AMT * P + tid]);
    int any_give = half_or(give, half);
    int base = 0, nb = 0;
    #pragma unroll 1
    for (int w2 = 0; w2 < (T >> 5); w2++) { int cw = wcnt[w2]; if (w2 < warp) base += cw; nb += cw; }
    if (mine) s_list[base + __popc(bm & ((1u << lane) - 1))] = tid;
    HSYNC();
    if (tid == 0 && (nb > 0 || any_give)) {
      #pragma unroll 1
      for (int i = nb - 1; i >= 1; i--) {
        int j = nm_bounded(draw(ctx, RS_BUY_SHUFFLE, (uint32_t)i, 0), i + 1);
        int t = s_list[i]; s_list[i] = s_list[j]; s_list[j] = t;
      }
      #pragma unroll 1
      for (int i = 0; i < nb; i++) { int p = s_list[i]; if (ent_alive(ctx, p)) act_buy(ctx, p, ctx.act[A_BUY * P + p]); }
      if (any_give) {
        #pragma unroll 1
        for (int p = 0; p < P; p++) if (ctx.act[A_GIVE_ITEM * P + p] && ent_alive(ctx, p)) act_give(ctx, p, ctx.act[A_GIVE_ITEM * P + p], ctx.act[A_GIVE_TARGET * P + p]);
        #pragma unroll 1
        for (int p = 0; p < P; p++) if (ctx.act[A_GOLD_AMT * P + p] && ent_alive(ctx, p)) act_give_gold(ctx, p, ctx.act[A_GOLD_AMT * P + p], ctx.act[A_GOLD_TARGET * P + p]);
      }
    }
    HSYNC();
  }
  PHASE();
  // Destroy (40)
  if (todo & 8) {
  #pragma unroll 1
  for (int p = tid; p < P; p += T) if (ent_alive(ctx, p) && ctx.act[A_DESTROY * P + p]) act_destroy(ctx, p, ctx.act[A_DESTROY * P + p]);
  HSYNC();
  }
  PHASE();
  // Attack (50): the reference executes attacks in entity-id order.  Two attacks commute unless
  // they share an entity (as attacker or target) or touch the item allocator (a kill, or the
  // last unit of ammunition).  The block therefore runs rounds: every pending attack registers its
  // index on both entities with atomicMin; an attack that holds the minimum on both is "ready";
  // ready attacks without allocator effects are applied in parallel, one per thread; an attack with
  // allocator effects is applied only when it is the lowest pending index, i.e. in exact
  // sequential position.  The lowest pending attack is always ready, so every round progresses.
  {
    const uint32_t DONE = 0xffffffffu;
    // pending attacks in attacker-row order (= the reference's execution order).  Every thread looks at its own
    // rows first: most ticks of a quiet environment have no attack at all and skip the ordered build.
    bool mine_any = false;
#pragma unroll
    for (int k = 0; k < V::kRowsPerThread; k++) {
      const int r = tid + k * T;
      int tgt = 0;
      if (r < P) tgt = ctx.act[A_ATT_TARGET * P + r]; else if (r < R) tgt = ctx.npc_att[r - P];
      mine_any |= tgt != 0 && tgt - 1 != r && ent_alive(ctx, r);
    }
    int *s_first2 = (int *)s_mv;                             // second registration array (the Move scratch is idle, >= R * 4 bytes)
    if (tid == 0) ctx.sc[6] = 0;
    if (half_or(mine_any, half)) {
      // ordered build by all warps: per-chunk counts, one barrier, each chunk writes at its prefix -- and registers
      // its attacks for round 0 in the same pass (the registration arrays are reset in the counting pass)
      int *s_cnt = (int *)s_scratch + 2 * R;
      const int n_chunks = (R + 31) >> 5;
      auto pending_target = [&](int r) -> int {
        int tgt = 0;
        if (r < P) tgt = ctx.act[A_ATT_TARGET * P + r]; else if (r < R) tgt = ctx.npc_att[r - P];
        return (tgt != 0 && tgt - 1 != r && ent_alive(ctx, r)) ? tgt : 0;
      };
      #pragma unroll 1
      for (int r = tid; r < R; r += T) { s_first[r] = 0x7fffffff; s_first2[r] = 0x7fffffff; }
      if (tid == 0) { ctx.sc[7] = 0x7fffffff; ctx.sc[24] = 0x7fffffff; }
      #pragma unroll 1
      for (int ch = warp; ch < n_chunks; ch += (T >> 5)) {
        const unsigned m = __ballot_sync(0xffffffffu, pending_target(ch * 32 + lane) != 0);
        if (lane == 0) s_cnt[ch] = __popc(m);
      }
      HSYNC();
      const int tag0 = ((1 << (31 - kIdxBits)) - 1) << kIdxBits;
      #pragma unroll 1
      for (int ch = warp; ch < n_chunks; ch += (T >> 5)) {
        int mine = 0, mine_before = 0;      // this lane's share of the per-chunk counts: chunks lane, lane + 32, ...
#pragma unroll
        for (int q = 0; q < V::kChunkIters; q++) {
          const int cq = lane + 32 * q, v = cq < n_chunks ? s_cnt[cq] : 0;
          mine += v; mine_before += cq < ch ? v : 0;
        }
        const int before = __reduce_add_sync(0xffffffffu, mine_before);
        const int r = ch * 32 + lane, tgt = pending_target(r);
        const unsigned m = __ballot_sync(0xffffffffu, tgt != 0);
        if (tgt) {
          const int i = before + __popc(m & ((1u << lane) - 1));
          s_att[i] = ((uint32_t)r << 16) | (uint32_t)(tgt - 1);
          atomicMin(&s_first[r], tag0 | i);
          atomicMin(&s_first[tgt - 1], tag0 | i);
        }
        // the lowest pending index of the chunk is its first attack; chunk 0 .. the first non-empty chunk holds index 0
        if (m && lane == 0) atomicMin(&ctx.sc[7], tag0 | before);
        if (ch == 0) { const int tot = __reduce_add_sync(0xffffffffu, mine); if (lane == 0) ctx.sc[6] = tot; }
      }
    }
    HSYNC();
    const int na = ctx.sc[6];
    int pending = na > 0;
    PCOUNT(22, na);
    // Rounds with one barrier each.  Registrations carry a round tag that shrinks from round to round, so a later
    // round's values undercut whatever earlier rounds left behind and nothing is ever cleared; and a round registers
    // its leftovers for the next round into the *other* of two registration arrays while its own is still being
    // checked (na < 2^kIdxBits attacks, fewer than 2^(31 - kIdxBits) rounds).
    int round = 0;
    #pragma unroll 1
    while (pending) {
      PCOUNT(23, 1);
      int *cur = (round & 1) ? s_first2 : s_first, *nxt = (round & 1) ? s_first : s_first2;
      int *low_cur = &ctx.sc[(round & 1) ? 24 : 7], *low_nxt = &ctx.sc[(round & 1) ? 7 : 24];
      const int tag = ((1 << (31 - kIdxBits)) - 1 - round) << kIdxBits, tag_n = ((1 << (31 - kIdxBits)) - 2 - round) << kIdxBits;
      round++;
      long long ta2 = clock64();
      const int lowest = *low_cur & ((1 << kIdxBits) - 1);
      int still = 0, my_low = 0x7fffffff;
      #pragma unroll 1
      for (int i = lane * (T >> 5) + warp; i < na; i += T) {
        uint32_t x = s_att[i];
        if (x == DONE) continue;
        int a = x >> 16, t = x & 0xffff;
        bool done = false;
        if (cur[a] == (tag | i) && cur[t] == (tag | i)) {
          done = true;
          if (ent_alive(ctx, a)) {
            int style = a < P ? (int)ctx.act[A_ATT_STYLE * P + a] : (int)ENT(EA_NPC_STYLE, a);
            int dmg; bool ammo_out;
            if (attack_compute(ctx, a, style, t, dmg, ammo_out)) {
              bool heavy = ammo_out || dmg >= ENT(EA_HEALTH, t);
              if (!heavy || i == lowest) attack_apply(ctx, a, style, t, dmg);
              else done = false;
            }
          }
        }
        if (done) s_att[i] = DONE;
        else {      // still pending: register for the next round right away
          still = 1;
          atomicMin(&nxt[a], tag_n | i);
          atomicMin(&nxt[t], tag_n | i);
          my_low = min(my_low, tag_n | i);
        }
      }
      my_low = __reduce_min_sync(0xffffffffu, my_low);
      if (lane == 0 && my_low != 0x7fffffff) atomicMin(low_nxt, my_low);
      pending = half_or(still, half);
      PCOUNT(46, clock64() - ta2);
    }
  }
  // VSmall4: the position index takes over the scratch (every read of the attack list is behind the last barrier above)
  #pragma unroll 1
  for (int i = tid; i < (V::kScratchInWs ? V::kTblSlots : 0); i += T) s_tbl[i] = 0;
  HSYNC();
  PHASE();
  // Move (60): with one entity per tile the reference resolves moves in entity-id order.
  if (c[NC_ALLOW_OCCUPIED]) {
    #pragma unroll 1
    for (int r = tid; r < R; r += T) if (ent_alive(ctx, r)) act_move(ctx, r, r < P ? (int)ctx.act[A_MOVE * P + r] : (int)ctx.npc_move[r - P], false);
  } else {
    // Sequential semantics: movers act in row order and a move succeeds iff the destination is
    // unoccupied at that moment.  With one entity per tile a destination d has at most four
    // claimants (one per neighbouring tile) and at most one occupant o, so every mover can decide
    // locally, from a position index (tile -> row), whether it is the one claimant that may take d:
    //   d free at tick start      -> the lowest-row claimant wins, the others find it occupied;
    //   d held by a mover o       -> claimants below o fail (o is still there); the first claimant
    //                                above o wins iff o itself moves away;
    //   d held by a non-mover     -> everybody fails.
    // The only non-local part is "iff o moves away": a chain of strictly decreasing rows that each
    // winner walks down.  No rounds, no atomics on the decision path.
    constexpr int KR = V::kRowsPerThread;
    constexpr unsigned TM = (unsigned)(V::kTblSlots - 1);
    const uint32_t NONE = 0xffffu, NODEP = 0xfffeu;          // verdict codes (rows are < 0xfffe)
    const tile_t NOTILE = (tile_t)~(tile_t)0;                // "does not move"
    uint32_t *tbl = s_tbl;                                   // position index, zeroed at the start of the tick: (tile + 1) << 12 | row
    tile_t *mvd = (tile_t *)s_mv;                            // intended destination
    uint16_t *res = (uint16_t *)(s_mv + (size_t)R * sizeof(tile_t));      // verdict / dependency
    int mv_dir[KR], mv_r[KR], mv_c[KR];                      // direction and destination (row, col)
#pragma unroll
    for (int k = 0; k < KR; k++) {
      int r = tid + k * T;
      mv_dir[k] = -1; mv_r[k] = 0; mv_c[k] = 0;
      if (r < R) {
        tile_t d = NOTILE;
        if (ent_alive(ctx, r)) {
          int dir = r < P ? (int)ctx.act[A_MOVE * P + r] : (int)ctx.npc_move[r - P];
          if (dir >= 0 && dir <= 3 && ENT(EA_FREEZE, r) == 0) {
            int nr = ENT(EA_ROW, r) + c_dir_dr[dir], nc = ENT(EA_COL, r) + c_dir_dc[dir];
            int dst = nr * S + nc;
            if (!nm_impassible(tile_i(ctx, dst))) { d = (tile_t)dst; mv_dir[k] = dir; mv_r[k] = nr; mv_c[k] = nc; }
          }
        }
        mvd[r] = d;
        if (ENT(EA_STATUS, r) == ES_ALIVE) {                 // position index: same set as the occupancy bitmap
          uint32_t key = (uint32_t)(ENT(EA_ROW, r) * S + ENT(EA_COL, r));
          uint32_t v = ((key + 1) << 12) | (uint32_t)r;
          unsigned h = (key * 40503u >> 3) & TM;
          while (atomicCAS(&tbl[h], 0u, v) != 0u) h = (h + 1) & TM;
        }
      }
    }
    HSYNC();
    auto who = [&](int tile) -> int {                        // row of the entity on an occupied tile
      unsigned h = ((unsigned)tile * 40503u >> 3) & TM;
      for (;;) {
        uint32_t cur = tbl[h];
        if ((cur >> 12) == (uint32_t)tile + 1) return (int)(cur & 0xfffu);
        if (cur == 0) return -1;
        h = (h + 1) & TM;
      }
    };
#pragma unroll
    for (int k = 0; k < KR; k++) {
      const int i = tid + k * T;
      if (mv_dir[k] < 0) { if (i < R) res[i] = (uint16_t)NONE; continue; }
      const int dr_ = mv_r[k], dc_ = mv_c[k], d = dr_ * S + dc_;
      // occupancy of the destination and of its other three neighbours first (five independent loads, no branches):
      // on a sparse map nearly every mask is empty and no index look-up happens at all
      const bool od = occ_get(ctx, dr_, dc_);
      unsigned nb = 0;
#pragma unroll
      for (int q = 0; q < 4; q++)
        if (q != mv_dir[k] && occ_get(ctx, dr_ - c_dir_dr[q], dc_ - c_dir_dc[q])) nb |= 1u << q;      // q == my direction: my own tile
      int o = od ? who(d) : -1;
      uint32_t verdict = NODEP;
      int lo = -1;                                           // claimants in (lo, i) beat me
      if (o >= 0) {
        if (mvd[o] == NOTILE || o > i) verdict = NONE; else { verdict = (uint32_t)o; lo = o; }
      }
      if (verdict != NONE) {
        #pragma unroll 1
        while (nb) {
          const int q = __ffs(nb) - 1; nb &= nb - 1;
          int e = who((dr_ - c_dir_dr[q]) * S + dc_ - c_dir_dc[q]);
          if (e > lo && e < i && mvd[e] == (tile_t)d) { verdict = NONE; break; }
        }
      }
      res[i] = (uint16_t)verdict;
    }
    HSYNC();
    bool mv_ok[KR];
#pragma unroll
    for (int k = 0; k < KR; k++) {
      mv_ok[k] = false;
      if (mv_dir[k] < 0) continue;
      int j = tid + k * T;
      for (;;) {
        uint32_t v = res[j];
        if (v == NONE) break;
        if (v == NODEP) { mv_ok[k] = true; break; }
        j = (int)v;
      }
      if (mv_ok[k]) occ_clr(ctx, ENT(EA_ROW, tid + k * T), ENT(EA_COL, tid + k * T));
    }
    HSYNC();
#pragma unroll
    for (int k = 0; k < KR; k++)
      if (mv_ok[k]) {
        occ_set(ctx, mv_r[k], mv_c[k]);
        act_move(ctx, tid + k * T, mv_dir[k], false);
      }
  }
  HSYNC();
  PHASE();
  // Sell (70)
  if (todo & 16) {
  #pragma unroll 1
  for (int p = tid; p < P; p += T) if (ent_alive(ctx, p) && ctx.act[A_SELL_ITEM * P + p]) act_sell(ctx, p, ctx.act[A_SELL_ITEM * P + p], ctx.act[A_SELL_PRICE * P + p]);
  HSYNC();
  }

  PHASE();
  // ---- phase 4: cull ------------------------------------------------------------------
  #pragma unroll 1
  for (int p = tid; p < P; p += T)
    if (ENT(EA_STATUS, p) == ES_ALIVE && ENT(EA_HEALTH, p) <= 0) {
      ENT(EA_STATUS, p) = ES_DEAD_THIS_TICK;
      occ_clr(ctx, ENT(EA_ROW, p), ENT(EA_COL, p));
      #pragma unroll 1
      while (ctx.invn[p] > 0) item_destroy(ctx, ctx.inv[p * NINV + ctx.invn[p] - 1]);
    }
  int *s_free = (int *)s_scratch + 512, *s_dng = (int *)s_scratch + 544;   // spawn inputs (scratch is idle here)
  {
    // NPC cull: every warp classifies 32-row chunks (dead now / still alive / free afterwards) and publishes the
    // three counts; after one barrier each chunk knows how many dead and free rows precede it, which gives the
    // danger-stack slot of every dead NPC (stack order = row order) and the ascending list of free rows.
    int *s_cnt = (int *)s_scratch + 600;                     // one packed count per chunk (<= 32 * kChunkIters chunks)
    const int n_chunks = (N + 31) >> 5;
    auto classify = [&](int r, bool &dead, bool &stays, bool &fr) {
      const bool live = r < R && ENT(EA_STATUS, r) == ES_ALIVE;
      dead = live && ENT(EA_HEALTH, r) <= 0;
      stays = live && !dead;
      fr = r < R && !stays;
    };
    #pragma unroll 1
    for (int ch = warp; ch < n_chunks; ch += (T >> 5)) {
      bool dead, stays, fr;
      classify(P + ch * 32 + lane, dead, stays, fr);
      const unsigned m = __ballot_sync(0xffffffffu, dead), am = __ballot_sync(0xffffffffu, stays), fm = __ballot_sync(0xffffffffu, fr);
      if (lane == 0) s_cnt[ch] = __popc(m) | (__popc(am) << 8) | (__popc(fm) << 16);
    }
    const int nd0 = ctx.sc[2];                               // read before the barrier: warp 0 replaces it below
    HSYNC();
    int16_t *danger = prm.danger + (size_t)env * N;
    #pragma unroll 1
    for (int ch = warp; ch < n_chunks; ch += (T >> 5)) {
      int dead_b = 0, free_b = 0, dead_all = 0, alive_all = 0;      // this lane's share: chunks lane, lane + 32, ...
#pragma unroll
      for (int q = 0; q < V::kChunkIters; q++) {
        const int cq = lane + 32 * q, v = cq < n_chunks ? s_cnt[cq] : 0;
        dead_all += v & 255; alive_all += (v >> 8) & 255;
        if (cq < ch) { dead_b += v & 255; free_b += (v >> 16) & 255; }
      }
      const int dead_before = __reduce_add_sync(0xffffffffu, dead_b), free_before = __reduce_add_sync(0xffffffffu, free_b);
      const int r = P + ch * 32 + lane;
      bool dead, stays, fr;
      classify(r, dead, stays, fr);
      const unsigned m = __ballot_sync(0xffffffffu, dead), fm = __ballot_sync(0xffffffffu, fr), lt = (1u << lane) - 1u;
      if (fr) { const int k = free_before + __popc(fm & lt); if (k < 32) s_free[k] = r; }      // the rows npcs.spawn will fill
      if (dead) {
        const int idx = nd0 + dead_before + __popc(m & lt);
        if (idx < N) danger[idx] = ENT(EA_NPC_DANGER, r);
        ENT(EA_STATUS, r) = ES_EMPTY;
        occ_clr(ctx, ENT(EA_ROW, r), ENT(EA_COL, r));
      }
      if (ch == 0) {
        const int tot_dead = __reduce_add_sync(0xffffffffu, dead_all), tot_alive = __reduce_add_sync(0xffffffffu, alive_all);
        if (lane == 0) { ctx.sc[2] = min(N, nd0 + tot_dead); ctx.sc[4] = tot_alive; }
      }
    }
  }
  HSYNC();
  PHASE();
  // ---- phase 5: npcs.spawn (sequential attempts) --------------------------------------
  const bool my_spawn = ctx.sc[4] < N;        // env-uniform: some NPC slot is free
  if (warp == (T >> 5) - 1) {      // the last warp has no part in the spawn draws: it finds the new high-water mark
    // of the item table meanwhile (no row is allocated or freed after the cull); read by the write-back
    int hi = 0;
    #pragma unroll 1
    for (int w0 = 0; w0 < cap_words; w0 += 32) {
      uint32_t u = w0 + lane < cap_words ? ctx.used[w0 + lane] : 0u;
      unsigned nz = __ballot_sync(0xffffffffu, u != 0);
      if (nz) { int top = 31 - __clz(nz); uint32_t ut = __shfl_sync(0xffffffffu, u, top); hi = ((w0 + top) << 5) + 32 - __clz(ut); }
    }
    if (lane == 0) ctx.sc[9] = (hi + 7) & ~7;
  }
  if (my_spawn) {
    // the draws of every attempt are keyed by (attempt, ordinal): compute them all in parallel
    const int n_pre = min(c[NC_NPC_SPAWN_ATTEMPTS] * 8, (int)(scratch_bytes / 4));
    if (my_spawn) for (int i = tid; i < n_pre; i += T) s_scratch[i] = draw(ctx, RS_NPC_SPAWN, (uint32_t)(i >> 3), (uint32_t)(i & 7));
    if (my_spawn && tid < 32) { int k = ctx.sc[2] - 1 - tid; s_dng[tid] = k >= 0 ? (int)prm.danger[(size_t)env * N + k] : 0; }   // top of the danger stack
    ctx.predraw = s_scratch;
    uint32_t *dec = s_scratch + 256;
    HSYNC();
    if (my_spawn && tid < 32) { const int n_acc = npc_spawn_decide(ctx, dec, s_free, s_dng, lane); if (tid == 0) ctx.sc[5] = n_acc; }
    HSYNC();
    if (my_spawn && tid < ctx.sc[5]) npc_spawn_fill(ctx, dec + tid * 8);
  }
  HSYNC();

  PHASE();
  // ---- phase 6: tick += 1, map.step, exchange.step ------------------------------------
  ctx.tick += 1;
  {
    // map.step: every depleted tile draws once.  Depleted tiles are first gathered into a
    // worklist (the draw is keyed by the tile, so order is free), then hashed by all threads
    tile_t *wl = (tile_t *)s_scratch;
    const int wl_cap = (int)(scratch_bytes / sizeof(tile_t));
    const int n_quads = S * S / 32;        // 16 bytes = 32 tiles per load
    auto respawn_tile = [&](int i, int m) {
      int thr_idx = m == MT_SCRUB ? NC_RESPAWN_FOILAGE : m == MT_SLAG ? NC_RESPAWN_ORE : m == MT_STUMP ? NC_RESPAWN_TREE
                  : m == MT_FRAGMENT ? NC_RESPAWN_CRYSTAL : m == MT_WEEDS ? NC_RESPAWN_HERB : NC_RESPAWN_FISH;
      if (draw(ctx, RS_RESPAWN, (uint32_t)i, 0) < (uint32_t)c.p[thr_idx]) tile_inc(ctx, i);
    };
    // The depleted tiles are known: the list carried over from last tick plus this tick's harvests (tile_dec).
    // Only when the list is unknown (first use after an overflow) is the map scanned to rebuild it.
    const bool list_ok = !prm.no_depl_list && n_depl0 >= 0 && ctx.sc[17] <= V::kDeplCap;
    // sc[19] (survivors) and sc[20] (scan hits) are still zero from the start of the tick: no set-up barrier
    if (!list_ok) {
    // depleted materials are 3, 6 and the even ones from 8 up: bit-sliced test of all 8 nibbles of a word
    auto hits_of = [](uint32_t x) -> uint32_t {
      const uint32_t x1 = x >> 1, x2 = x >> 2, x3 = x >> 3;
      return ((x3 & ~x) | (~x3 & x1 & (x2 ^ x))) & 0x11111111u;
    };
    // pass 1 counts this thread's hits over all its quads, one scan + one shared-memory atomic per warp reserves
    // the worklist slots, pass 2 re-tests the same words (cheaper than keeping the masks) and fills them in
    int cnt = 0;
    #pragma unroll 1
    for (int q = tid; q < n_quads; q += T) {
      const uint4 v = ((const uint4 *)ctx.map)[q];
      cnt += __popc(hits_of(v.x)) + __popc(hits_of(v.y)) + __popc(hits_of(v.z)) + __popc(hits_of(v.w));
    }
    if (__any_sync(0xffffffffu, cnt)) {
      int incl = cnt;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += u; }
      int base = 0;
      if (lane == 31) base = atomicAdd(&ctx.sc[20], incl);
      int k = __shfl_sync(0xffffffffu, base, 31) + incl - cnt;
      if (cnt)
        #pragma unroll 1
        for (int q = tid; q < n_quads; q += T) {
          const uint4 v = ((const uint4 *)ctx.map)[q];
          const uint32_t xs[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int j = 0; j < 4; j++) {
            uint32_t hit = hits_of(xs[j]);
            #pragma unroll 1
            while (hit) {
              int b = __ffs(hit) - 1; hit &= hit - 1;
              int i = (q * 4 + j) * 8 + (b >> 2);
              if (k < wl_cap) wl[k] = (tile_t)i;
              else respawn_tile(i, tile_i(ctx, i));          // worklist full: draw in place
              k++;
            }
          }
        }
    }
    HSYNC();
    }
    const tile_t *src = list_ok ? ctx.dlist : wl;
    tile_t *dst = list_ok ? wl : ctx.dlist;
    const int n_src = list_ok ? ctx.sc[17] : min(ctx.sc[20], wl_cap), dst_cap = list_ok ? wl_cap : V::kDeplCap;
    // Fold the tick's events here (nothing emits after the spawn): the last threads fold while the first ones
    // walk the depleted tiles below, and the fold's global atomics -- one returns a value -- are in flight
    // underneath the walk.  The barriers that follow order them before the reward phase reads the counters.
    {
      const int nev = min(ctx.sc[0], prm.ev_cap);
      PCOUNT(26, nev);
      uint2 *const ev_log = prm.ev_log ? prm.ev_log + (size_t)env * prm.ev_cap : nullptr;      // event log on: keep the ring
      if (ev_log && tid == 0) prm.ev_n[env] = nev;
      #pragma unroll 1
      for (int i = T - 1 - tid; i < nev; i += T) {
        const uint2 e = ctx.ev[i];
        if (ev_log) ev_log[i] = e;
        fold_event(ctx, e);
      }
    }
    // one draw per depleted tile; the tiles that stay depleted form next tick's list
    #pragma unroll 1
    for (int k0 = 0; k0 < n_src; k0 += T) {
      const int k = k0 + tid;
      bool stays = false;
      int i = 0;
      if (k < n_src) {
        i = src[k];
        const int m = tile_i(ctx, i);
        const int thr_idx = m == MT_SCRUB ? NC_RESPAWN_FOILAGE : m == MT_SLAG ? NC_RESPAWN_ORE : m == MT_STUMP ? NC_RESPAWN_TREE
                          : m == MT_FRAGMENT ? NC_RESPAWN_CRYSTAL : m == MT_WEEDS ? NC_RESPAWN_HERB : NC_RESPAWN_FISH;
        if (draw(ctx, RS_RESPAWN, (uint32_t)i, 0) < (uint32_t)c.p[thr_idx]) tile_inc(ctx, i); else stays = true;
      }
      const unsigned sm = __ballot_sync(0xffffffffu, stays);
      int base = 0;
      if (lane == 0 && sm) base = atomicAdd(&ctx.sc[19], __popc(sm));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (stays) { const int pos = base + __popc(sm & ((1u << lane) - 1)); if (pos < dst_cap) dst[pos] = (tile_t)i; }
    }
    HSYNC();
    if (tid == 0) {
      const bool scan_overflow = !list_ok && ctx.sc[20] > wl_cap;      // tiles beyond the worklist drew in place and are not listed
      ctx.sc[21] = (ctx.sc[19] <= min(V::kDeplCap, dst_cap) && !scan_overflow) ? ctx.sc[19] : -1;
      ctx.sc[22] = list_ok ? 0 : 1;                                    // which buffer holds the new list: worklist scratch / dlist
    }
  }
  // rows the table grew over this tick that are not in use must read as empty from now on
  #pragma unroll 1
  for (int r = item_hi0 + tid; r < ctx.sc[9]; r += T)
    if (!row_used(ctx, r)) {
#pragma unroll
      for (int k = 0; k < IS_N; k++) ITM(k, r) = 0;
    }
  // exchange.step: listings expire; only rows in use are visited.  One row per thread: rows are allocated lowest-first,
  // so the live ones share a bitmap word or two, and with the item table in place (HBM / L2) a thread that walked a whole
  // word paid two dependent L2 round trips per row, one row after the other (9 K cycles per env-tick in the driver's window)
  #pragma unroll 1
  for (int i = tid; i < ctx.sc[9]; i += T)
    if (row_used(ctx, i)) {
      const int price = ITM(IS_PRICE, i), listed_at = ITM(IS_LIST_TICK, i);
      if (price > 0 && ctx.tick - listed_at > c[NC_LISTING_DURATION]) { ITM(IS_PRICE, i) = 0; ITM(IS_LIST_TICK, i) = 0; }
    }
  HSYNC();

  PHASE();
  // ---- write the tables back while the wrapper part runs ------------------------------
  if (!V::kGlobalTables) {
  fence_async_smem();
  HSYNC();
  if (tid == 0) {
    bulk_s2g(prm.ent + (size_t)env * EA_N * R, ctx.ent, ent_bytes);
    const int hi = ctx.sc[9];
    const uint32_t col_bytes = (uint32_t)hi * 2;
    if (col_bytes && !V::kItemsInPlace)
      for (int k = 0; k < IS_N; k++) bulk_s2g(gitem + (size_t)k * CAP, ctx.item + k * CAP, col_bytes);
    bulk_s2g(prm.map + (size_t)env * map_bytes, ctx.map, map_bytes);
    if (ctx.sc[21] > 0 && !(kDeplInPlace && ctx.sc[22]))      // (in place: a list rebuilt into dlist is already there)
      bulk_s2g(gdepl, ctx.sc[22] ? (const void *)ctx.dlist : (const void *)s_scratch, (uint32_t)((ctx.sc[21] * (int)sizeof(tile_t) + 15) & ~15));
    bulk_commit();
  }
  } else {
    // the tables are already where they live; only a list that ended up in the shared-memory worklist moves
    if (ctx.sc[21] > 0 && !ctx.sc[22]) {
      const tile_t *wl2 = (const tile_t *)s_scratch;
      #pragma unroll 1
      for (int i = tid; i < ctx.sc[21]; i += T) gdepl[i] = wl2[i];
    }
    HSYNC();      // the scratch is reused by the reward phase
  }

  PHASE();
  // ---- phase 7: (the tick's events were folded before phase 6) --------------------------

  PHASE();
  // ---- phase 8: rewards, done flags, stat wrapper --------------------------------------
  int st_me = tid < P ? (int)ENT(EA_STATUS, tid) : ES_EMPTY;
  // window-scan predicates (CanSeeTile / CanSeeAgent / CanSeeGroup) are evaluated by a whole warp
  // per requesting agent instead of a 225- or 384-iteration loop in one lane
  // requesting agents are gathered into a list (s_list is idle here) that all warps share out
  if (tid == 0) ctx.sc[18] = 0;
  HSYNC();
  {
    bool req = tid < P && st_me == ES_ALIVE && !my_done && my_t[4] == 0 && (my_t[0] == TP_CAN_SEE_TILE || my_t[0] == TP_CAN_SEE_AGENT || my_t[0] == TP_CAN_SEE_GROUP);
    if (tid < P) ctx.slow[tid] = (int8_t)-1;
    unsigned rm = __ballot_sync(0xffffffffu, req);
    int wbase = 0;
    if (lane == 0 && rm) wbase = atomicAdd(&ctx.sc[18], __popc(rm));
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    if (req) s_list[wbase + __popc(rm & ((1u << lane) - 1))] = tid;
  }
  HSYNC();
  {
  const int n_req = ctx.sc[18];
  #pragma unroll 1
  for (int qi = warp; qi < n_req; qi += (T >> 5)) {
    const int p = s_list[qi];
    int pred = ctx.task[p * 4], q0 = ctx.task[p * 4 + 1], q1 = ctx.task[p * 4 + 2];
    int r = ENT(EA_ROW, p), cc = ENT(EA_COL, p), vis = c[NC_VISION];
    bool hit = false;
    if (pred == TP_CAN_SEE_TILE) {
      int win = 2 * vis + 1;
      #pragma unroll 1
      for (int w = lane, dr = lane / win, dc = lane % win; w < win * win; w += 32) {      // (dr, dc) advance without dividing
        hit |= tile_at(ctx, r - vis + dr, cc - vis + dc) == q0;
        dr += 32 / win; dc += 32 % win;
        if (dc >= win) { dc -= win; dr++; }
      }
      hit = __any_sync(0xffffffffu, hit);
    } else {
      int lo = q0, hi = pred == TP_CAN_SEE_AGENT ? q0 : q1, seen = 0;
      #pragma unroll 1
      const int n_ent_obs = V::kStd ? kStdL.n_ent : prm.L.n_ent;
      for (int base = 0; base < R && seen < n_ent_obs; base += 32) {
        int row = base + lane;
        bool in = row < R && ENT(EA_STATUS, row) == ES_ALIVE && nm_iabs(ENT(EA_ROW, row) - r) <= vis && nm_iabs(ENT(EA_COL, row) - cc) <= vis;
        unsigned bm = __ballot_sync(0xffffffffu, in);
        int rank = seen + __popc(bm & ((1u << lane) - 1));
        int id = in ? (int)ENT(EA_ID, row) : 0;
        hit |= in && rank < n_ent_obs && id >= lo && id <= hi;
        seen += __popc(bm);
      }
      hit = __any_sync(0xffffffffu, hit);
    }
    if (lane == 0) ctx.slow[p] = hit ? 1 : 0;
  }
  }
  HSYNC();
  PHASE();
  int n_alive = half_count(st_me == ES_ALIVE, half);
  int n_dead = half_count(st_me == ES_DEAD_THIS_TICK, half);
  int n_current = n_alive + n_dead;
  bool horizon = ctx.tick >= c[NC_HORIZON];
  if (horizon) n_current = 0;
  bool env_done = n_current <= c[NC_EARLY_STOP_N] || n_alive == 0;
  if (tid < P) {       // P <= blockDim: one thread per player, state prefetched at kernel start
    const int p = tid;
    const size_t a = my_a;
    int st = st_me;
    float rew = 0.0f; uint8_t term = 0, trunc = 0, mask = 0;
    prm.info_valid[a] = 0;
    if (st != ES_EMPTY) {
      mask = 1;
      bool terminated = st == ES_DEAD_THIS_TICK;
      bool truncated = horizon && !terminated;
      double reward;
      int completed = my_done, signals = my_signals;
      int acc0 = ctx.acc[p * 2], acc1 = ctx.acc[p * 2 + 1];
      if (acc0 != my_acc0) my_sta[ST_TASK_ACC0] = acc0;
      if (acc1 != my_acc1) my_sta[ST_TASK_ACC1] = acc1;
      if (terminated) reward = -1.0;
      else {
        double diff = 0.0;
        if (!completed) {
          double v;
          if (my_t[4]) {
            // team subject / named target (nm_task_flag): rare; one inlined copy instead of a flag test in every predicate
            v = flagged_task_value(ctx, p, make_int4(my_t[0], my_t[1], my_t[2], my_t[3]), make_int4(my_t[4], my_t[5], my_t[6], my_t[7]),
                                   make_int4(my_t[8], my_t[9], my_t[10], my_t[11]), acc0, acc1);
          } else {
          v = eval_predicate(ctx, p, my_t[0], my_t[1], my_t[2], my_t[3], acc0, acc1);
          if (my_t[7] == 1) v = v * eval_predicate(ctx, p, my_t[5], my_t[6], my_t[8], my_t[9], 0, 0);
          else if (my_t[7] == 2)      // (wa/1000) * a + (wb/1000) * b, each operation rounded like the reference's Python floats
            v = __dadd_rn(__dmul_rn(__ddiv_rn((double)my_t[10], 1000.0), v),
                          __dmul_rn(__ddiv_rn((double)my_t[11], 1000.0), eval_predicate(ctx, p, my_t[5], my_t[6], my_t[8], my_t[9], 0, 0)));
          }
          v = clip01(v);
          diff = v - my_prog;
          if (v != my_prog) my_ds[DS_PROGRESS] = v;
          my_prog = v;
          if (v >= 1.0) { completed = ctx.tick; my_sta[ST_TASK_DONE] = completed; }
        }
        reward = diff;
        if (reward > 0) { signals++; my_sta[ST_REWARD_SIGNALS] = signals; }
        if (my_prog > my_maxprog) { my_maxprog = my_prog; my_ds[DS_MAX_PROGRESS] = my_maxprog; }
      }
      if (env_done && !terminated) truncated = true;
      int uprev = my_uniq, ucurr = uprev + ctx.duniq[p];
      my_sta[ST_UNIQ_PREV] = uprev;
      if (ucurr != uprev) my_sta[ST_UNIQ_CURR] = ucurr;
      if (!(terminated || truncated)) { if (reward != 0.0) my_ds[DS_CUM_REWARD] = my_cum + reward; }
      else write_info(ctx, p, terminated, my_cum, my_maxprog, signals, completed, ucurr);
      if (c[NC_USE_CUSTOM_REWARD]) {
        double explore = 0.0;
        if (prm.fcfg[NF_EXPLORE_W] > 0 && ucurr > uprev) explore = (double)min(c[NC_CLIP_UNIQUE], ucurr - uprev) * prm.fcfg[NF_EXPLORE_W];
        if (c[NC_WRAPPER] == NW_TAKERU) { if (!(terminated || truncated)) reward += explore; }
        else if (c[NC_WRAPPER] == NW_START_KIT) {
          double heal = 0.0;
          if (prm.fcfg[NF_HEAL_W] > 0 && st == ES_ALIVE && ENT(EA_HEALTH_RESTORE, p) > 0) heal = prm.fcfg[NF_HEAL_W];
          reward += heal + explore;
        } else if (c[NC_WRAPPER] == NW_YAOFENG) {
          // yaofeng/reward_wrapper.py:85-129: deltas of hp / best skill exp / damage inflicted / gold since the
          // agent's previous tick plus the equipment defense term, in the reference's operation order
          // (explicit round-to-nearest multiplies and adds: no fused multiply-add)
          if (!(terminated || truncated)) {
            const int hp = ENT(EA_HEALTH, p), gold = ENT(EA_GOLD, p), dmg = ENT(EA_DMG_INFLICTED, p);
            int cur_exp = 0;
            #pragma unroll 1
            for (int col = EA_MELEE_EXP; col <= EA_ALCHEMY_EXP; col += 2) cur_exp = max(cur_exp, (int)ENT(col, p));
            int def3 = 0;
            #pragma unroll 1
            for (int s2 = EA_EQ_HAT; s2 <= EA_EQ_AMMO; s2++) { int it = ENT(s2, p); if (it) def3 += 3 * item_defense(c, ITM(IS_TYPE, it - 1), ITM(IS_LEVEL, it - 1)); }
            const double hp_bonus = __dmul_rn((double)(hp - my_sta[ST_Y_HP]), prm.fcfg[NF_HP_W]);
            const double exp_bonus = __dmul_rn((double)(cur_exp - my_sta[ST_Y_EXP]), prm.fcfg[NF_EXP_W]);
            const double defense_bonus = __dmul_rn(prm.fcfg[NF_DEFENSE_W], __ddiv_rn((double)def3, 45.0));
            const double attack_bonus = __dmul_rn((double)(dmg - my_sta[ST_Y_DMG_INFLICTED]), prm.fcfg[NF_ATTACK_W]);
            const double gold_bonus = __dmul_rn((double)(gold - my_sta[ST_Y_GOLD]), prm.fcfg[NF_GOLD_W]);
            my_sta[ST_Y_HP] = hp; my_sta[ST_Y_EXP] = cur_exp; my_sta[ST_Y_DMG_INFLICTED] = dmg; my_sta[ST_Y_GOLD] = gold;
            double sum = __dadd_rn(hp_bonus, exp_bonus);
            sum = __dadd_rn(sum, defense_bonus); sum = __dadd_rn(sum, attack_bonus); sum = __dadd_rn(sum, gold_bonus);
            reward = __dadd_rn(reward, __dmul_rn(sum, prm.fcfg[NF_BONUS_SCALE]));
          }
        }
      } else if (terminated) reward = 0.0;
      rew = (float)reward; term = terminated; trunc = truncated;
    }
    prm.rew[a] = rew; prm.term[a] = term; prm.trunc[a] = trunc; prm.mask[a] = mask;
  }
  PHASE();
  PCOUNT(27, n_alive); PCOUNT(28, n_dead);
  if (tid == 0) {
    gsc[SC_TICK] = ctx.tick; gsc[SC_DONE] = env_done ? 1 : 0; gsc[SC_N_DANGER] = ctx.sc[2]; gsc[SC_NEXT_NPC_ID] = ctx.sc[3];
    gsc[SC_FRESH] = 0; gsc[SC_ITEM_HI] = ctx.sc[9]; gsc[SC_N_DEPL] = prm.no_depl_list ? -1 : ctx.sc[21];
    if (ctx.sc[1]) { gsc[SC_ERROR] |= 1; atomicAdd(&prm.counters[3], 1ULL); }
    prm.episode_done[env] = env_done ? 1 : 0;
    atomicAdd(&prm.counters[0], (unsigned long long)P);
    atomicAdd(&prm.counters[1], (unsigned long long)(n_alive + n_dead));
    if (!V::kGlobalTables) bulk_wait_all();
  }
  PHASE();
}
#undef half_or
#undef half_count

extern "C" __global__ void __launch_bounds__(2 * VSmall::kThreads, 1)
nmmo_step_kernel(const __grid_constant__ NmParams prm) { step_body<VSmall>(prm); }

extern "C" __global__ void __launch_bounds__(3 * VSmall3::kThreads, 1)
nmmo_step3_kernel(const __grid_constant__ NmParams prm) { step_body<VSmall3>(prm); }

extern "C" __global__ void __launch_bounds__(3 * VSmall3Std::kThreads, 1)
nmmo_step3_std_kernel(const __grid_constant__ NmParams prm) { step_body<VSmall3Std>(prm); }

extern "C" __global__ void __launch_bounds__(4 * VSmall4::kThreads, 1)
nmmo_step4_kernel(const __grid_constant__ NmParams prm) { step_body<VSmall4>(prm); }

extern "C" __global__ void __launch_bounds__(4 * VSmall4Std::kThreads, 1)
nmmo_step4_std_kernel(const __grid_constant__ NmParams prm) { step_body<VSmall4Std>(prm); }

extern "C" __global__ void __launch_bounds__(VBig::kThreads, 1)
nmmo_step_big_kernel(const __grid_constant__ NmParams prm) { step_body<VBig>(prm); }

extern "C" __global__ void __launch_bounds__(VBigStd::kThreads, 1)
nmmo_step_big_std_kernel(const __grid_constant__ NmParams prm) { step_body<VBigStd>(prm); }
