/*
 * nmmo_spec.h -- frozen constants and memory layout of the batched Neural MMO step.
 *
 * This header is pure data description (enums, column indices, record offsets). It is
 * shared by the CUDA product (nmmo_b200/csrc), the C-ABI (include/nmmo_b200.h) and the
 * CPU oracle (oracle/), exactly like a wire-format spec: it contains NO game arithmetic.
 *
 * Provenance.  The simulator the reference drives (`nmmo>=2.1,<2.2`,
 * /root/reference/pyproject.toml:19) is an un-vendored dependency that is absent from this
 * container, so every constant below that is not citable in /root/reference is a restatement
 * of upstream nmmo 2.1 from its published source layout (module names in comments) and is
 * tagged [UPSTREAM].  Constants evidenced in the reference itself carry a file:line.
 */
#ifndef NMMO_SPEC_H
#define NMMO_SPEC_H

#include <stdint.h>

#ifdef __CUDACC__
#define NM_HD __host__ __device__
#else
#define NM_HD
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------ config vector ---- */
/* The engine config travels as a flat int32 vector (no struct ABI issues across ctypes /
 * cgo / JNI).  Indices mirror reinforcement_learning/environment.py:14-49 (overrides) plus
 * the nmmo.core.config defaults [UPSTREAM]. */
enum nm_cfg {
  NC_N_PLAYERS = 0,      /* PLAYER_N            environment.py:33  (128) */
  NC_N_NPCS,             /* NPC_N               environment.py:43  (256) */
  NC_HORIZON,            /* HORIZON             environment.py:34  (1024) */
  NC_MAP_CENTER,         /* MAP_CENTER          environment.py:42  (128) */
  NC_MAP_BORDER,         /* MAP_BORDER          [UPSTREAM] 16 */
  NC_MAP_SIZE,           /* CENTER + 2*BORDER   manual_curriculum.py:152-154 (160) */
  NC_N_ENT_OBS,          /* PLAYER_N_OBS        [UPSTREAM] 100 */
  NC_N_MKT_OBS,          /* MARKET_N_OBS        [UPSTREAM] 384 */
  NC_N_INV,              /* ITEM_INVENTORY_CAPACITY   takeru/policy.py:264 (12) */
  NC_N_PRICE,            /* PRICE_N_OBS         takeru/policy.py:318,322 (99) */
  NC_VISION,             /* PLAYER_VISION_RADIUS      baseline_policy.py:96-97 (7) */
  NC_TASK_DIM,           /* TASK_EMBED_DIM      environment.py:44 (2048) */
  NC_NPC_VISION,         /* Entity.vision for NPCs [UPSTREAM] 5 */
  /* resources (nmmo.core.config.Resource) [UPSTREAM] */
  NC_RES_BASE,           /* 100 */
  NC_RES_DEPLETION,      /* 5 */
  NC_RES_STARVATION,     /* 10 */
  NC_RES_DEHYDRATION,    /* 10 */
  NC_RES_REGEN_THRESH,   /* floor(0.5 * base) = 50: regen when food>thresh && water>thresh */
  NC_RES_HEALTH_RESTORE, /* floor(0.1 * base) = 10 */
  NC_RES_HARVEST_RESTORE,/* floor(1.0 * base) = 100 */
  NC_RES_RESILIENT_N,    /* round(RESOURCE_RESILIENT_POPULATION * PLAYER_N) environment.py:45 */
  /* combat (nmmo.core.config.Combat) */
  NC_SPAWN_IMMUNITY,     /* COMBAT_SPAWN_IMMUNITY environment.py:46 (20) */
  NC_REACH,              /* 3 */
  NC_FREEZE_TIME,        /* COMBAT_STATUS_DURATION 3; takeru/policy.py:134 */
  NC_WEAK_NUM, NC_WEAK_DEN,       /* weakness multiplier 3/2 */
  NC_MINDMG_NUM, NC_MINDMG_DEN,   /* minimum damage proportion 1/4 */
  /* progression */
  NC_LEVEL_MAX,          /* 10  takeru/policy.py:128 */
  NC_XP_COMBAT, NC_XP_AMMO, NC_XP_CONSUMABLE,
  NC_BASE_DAMAGE, NC_LEVEL_DAMAGE, NC_BASE_DEFENSE, NC_LEVEL_DEFENSE,
  NC_EXP_THRESH0,        /* 10 entries: exp needed for level i+1 */
  NC_EXP_THRESH_LAST = NC_EXP_THRESH0 + 9,
  /* npc */
  NC_NPC_SPAWN_ATTEMPTS,
  NC_NPC_AGGR_PCT, NC_NPC_NEUT_PCT, NC_NPC_PASS_PCT,   /* danger thresholds, percent */
  NC_NPC_LEVEL_MIN, NC_NPC_LEVEL_MAX,
  NC_NPC_BASE_DEFENSE, NC_NPC_LEVEL_DEFENSE, NC_NPC_BASE_DAMAGE, NC_NPC_LEVEL_DAMAGE,
  /* equipment / items */
  NC_WEAPON_DROP_THR,    /* u32 threshold of WEAPON_DROP_PROB (0.025) */
  NC_WEAPON_BASE, NC_WEAPON_LEVEL, NC_AMMO_BASE, NC_AMMO_LEVEL,
  NC_TOOL_BASE, NC_TOOL_LEVEL, NC_ARMOR_BASE, NC_ARMOR_LEVEL,
  NC_RESTORE_BASE, NC_RESTORE_LEVEL,       /* consumable restore = 50 + 5*level */
  /* profession: respawn thresholds (u32 of probability), indexed by harvestable class */
  NC_RESPAWN_FOILAGE, NC_RESPAWN_ORE, NC_RESPAWN_TREE, NC_RESPAWN_CRYSTAL, NC_RESPAWN_HERB,
  NC_RESPAWN_FISH,
  /* exchange */
  NC_BASE_GOLD, NC_LISTING_DURATION,
  /* movement */
  NC_ALLOW_OCCUPIED,     /* ALLOW_MOVE_INTO_OCCUPIED_TILE (0 = one entity per tile) */
  /* wrapper (stat_wrapper.py:10-24, agent_zoo reward wrappers) */
  NC_WRAPPER,            /* nm_wrapper */
  NC_EARLY_STOP_N,       /* early_stop_agent_num  config.yaml:100,138 */
  NC_EVAL_MODE, NC_USE_CUSTOM_REWARD,
  NC_CLIP_UNIQUE,        /* clip_unique_event 3 */
  NC_DISABLE_GIVE,       /* takeru/reward_wrapper.py:31-35, yaofeng/reward_wrapper.py:72-76 */
  NC_NO_DANGEROUS_NPC,   /* donot_attack_dangerous_npc  yaofeng/reward_wrapper.py:78-81 */
  NC_ITEM_CAP,           /* item table rows = N_PLAYERS * N_INV */
  /* stress workload knobs (BASELINE.json configs[4]; no counterpart in the reference's Config: it only scales
   * PLAYER_N / NPC_N / MAP_CENTER, config.yaml:76-80) */
  NC_SPAWN_PATCH,        /* 0 = players spawn on the border ring; k > 0 = all players spawn inside a k x k patch
                            centred on the map ("clustered spawn"), k * k >= PLAYER_N */
  NC_TEAM_SIZE,          /* players per team (0 or 1 = every agent is its own team, the AgentTraining game of
                            environment.py:48); teams are consecutive id ranges, the first member is the leader */
  NC_SAMPLE_MOVE_PCT,    /* built-in action sampler only: percent probability that the Move head picks a valid
                            direction other than Stay (0 = uniform over the valid entries, config 2) */
  /* death fog (nmmo/entity/player.py Player.update) [UPSTREAM] */
  NC_DEATH_FOG,          /* PLAYER_DEATH_FOG: first tick of the fog, -1 = None (off)  config.yaml:75-86 death_fog_tick,
                            environment.py:36-39 */
  NC_DEATH_FOG_SPEED,    /* PLAYER_DEATH_FOG_SPEED 1: damage added per tick of fog */
  NC_DEATH_FOG_FINAL_SIZE,  /* PLAYER_DEATH_FOG_FINAL_SIZE 8: Chebyshev radius around the map centre the fog never enters */
  NC_COUNT
};

/* float config (double vector) */
enum nm_fcfg {
  NF_EXPLORE_W = 0,      /* explore_bonus_weight  config.yaml:105,139 */
  NF_HEAL_W,             /* heal_bonus_weight     config.yaml:104 */
  /* yaofeng/reward_wrapper.py:20-25, config.yaml:117-123 */
  NF_HP_W, NF_EXP_W, NF_DEFENSE_W, NF_ATTACK_W, NF_GOLD_W, NF_BONUS_SCALE,
  NF_COUNT
};

enum nm_wrapper { NW_BASE = 0, NW_TAKERU = 1, NW_START_KIT = 2, NW_YAOFENG = 3 };

/* --------------------------------------------------------------- entity table ------- */
/* Observed columns 0..30: EntityState [UPSTREAM nmmo/entity/entity.py]; the 31 names are
 * evidenced at agent_zoo/takeru/policy.py:120-161, count 31 at yaofeng/policy.py:141. */
enum nm_ent {
  EA_ID = 0, EA_NPC_TYPE, EA_ROW, EA_COL,
  EA_DAMAGE, EA_TIME_ALIVE, EA_FREEZE, EA_ITEM_LEVEL, EA_ATTACKER_ID, EA_LATEST_COMBAT_TICK,
  EA_MESSAGE,
  EA_GOLD, EA_HEALTH, EA_FOOD, EA_WATER,
  EA_MELEE_LEVEL, EA_MELEE_EXP, EA_RANGE_LEVEL, EA_RANGE_EXP, EA_MAGE_LEVEL, EA_MAGE_EXP,
  EA_FISHING_LEVEL, EA_FISHING_EXP, EA_HERBALISM_LEVEL, EA_HERBALISM_EXP,
  EA_PROSPECTING_LEVEL, EA_PROSPECTING_EXP, EA_CARVING_LEVEL, EA_CARVING_EXP,
  EA_ALCHEMY_LEVEL, EA_ALCHEMY_EXP,
  EA_N_OBS = 31,
  /* hidden columns (engine state that is not observed).  A row is either a player or an NPC,
   * so the NPC-only columns share storage with player-only columns. */
  EA_H0 = 31,
  EA_EXPLORATION = 31,   /* History.exploration (players) */
  EA_SPAWN_ROW, EA_SPAWN_COL,
  EA_HEALTH_RESTORE,     /* Resources.health_restore  start_kit/reward_wrapper.py:69 */
  EA_RESILIENT,
  EA_EQ_HAT, EA_EQ_TOP, EA_EQ_BOTTOM, EA_EQ_HELD, EA_EQ_AMMO,  /* item row + 1, 0 = empty (players) */
  EA_DMG_INFLICTED, EA_DMG_RECEIVED,                           /* History (players and NPCs) */
  EA_STATUS,             /* 0 empty row, 1 alive, 2 culled this tick (kept for episode stats) */
  EA_N = 44,
  /* NPC-only hidden state, aliased onto the player-only columns above */
  EA_NPC_STYLE = EA_EXPLORATION,        /* 0 melee 1 range 2 mage */
  EA_NPC_TARGET = EA_SPAWN_ROW,         /* entity id of hunt target, 0 none */
  EA_NPC_DANGER = EA_SPAWN_COL,         /* spawn distance-from-border d */
  EA_NPC_OFFENSE = EA_HEALTH_RESTORE, EA_NPC_DEFENSE = EA_RESILIENT,
  EA_NPC_DROP_ARMOR = EA_EQ_HAT, EA_NPC_DROP_TOOL = EA_EQ_TOP   /* item type ids */
};
enum nm_status { ES_EMPTY = 0, ES_ALIVE = 1, ES_DEAD_THIS_TICK = 2 };

/* ----------------------------------------------------------------- item table ------- */
/* ItemState [UPSTREAM nmmo/systems/item.py]; col 1 type, col 14 equipped evidenced at
 * neurips23_start_kit/baseline_policy.py:162-163; 16 columns at takeru/policy.py:223-241 */
enum nm_item {
  IA_ID = 0, IA_TYPE, IA_OWNER, IA_LEVEL, IA_CAPACITY, IA_QUANTITY,
  IA_MELEE_ATTACK, IA_RANGE_ATTACK, IA_MAGE_ATTACK,
  IA_MELEE_DEFENSE, IA_RANGE_DEFENSE, IA_MAGE_DEFENSE,
  IA_HEALTH_RESTORE, IA_RESOURCE_RESTORE, IA_EQUIPPED, IA_LISTED_PRICE,
  IA_N_OBS = 16
};
/* stored columns (the attack/defense/restore columns are pure functions of type+level) */
enum nm_item_store { IS_TYPE = 0, IS_LEVEL, IS_OWNER, IS_QUANTITY, IS_EQUIPPED, IS_PRICE,
                     IS_LIST_TICK, IS_N = 7 };

enum nm_item_type {   /* ITEM_TYPE_ID [UPSTREAM]; 18 classes 0..17 baseline_policy.py:163 */
  IT_NONE = 0, IT_GOLD = 1,
  IT_HAT = 2, IT_TOP = 3, IT_BOTTOM = 4,
  IT_SPEAR = 5, IT_BOW = 6, IT_WAND = 7,
  IT_ROD = 8, IT_GLOVES = 9, IT_PICKAXE = 10, IT_AXE = 11, IT_CHISEL = 12,
  IT_WHETSTONE = 13, IT_ARROW = 14, IT_RUNES = 15,
  IT_RATION = 16, IT_POTION = 17, IT_N = 18
};

/* ------------------------------------------------------------------ materials ------- */
enum nm_material {    /* nmmo/lib/material.py [UPSTREAM] */
  MT_VOID = 0, MT_WATER, MT_GRASS, MT_SCRUB, MT_FOILAGE, MT_STONE, MT_SLAG, MT_ORE,
  MT_STUMP, MT_TREE, MT_FRAGMENT, MT_CRYSTAL, MT_WEEDS, MT_HERB, MT_OCEAN, MT_FISH, MT_N
};
/* bit m set => material m impassible: Void, Water, Stone, Ocean, Fish */
#define NM_IMPASSIBLE_MASK ((1u<<MT_VOID)|(1u<<MT_WATER)|(1u<<MT_STONE)|(1u<<MT_OCEAN)|(1u<<MT_FISH))
/* depleted states: Scrub, Slag, Stump, Fragment, Weeds, Ocean (restore = state + 1) */
#define NM_DEPLETED_MASK ((1u<<MT_SCRUB)|(1u<<MT_SLAG)|(1u<<MT_STUMP)|(1u<<MT_FRAGMENT)|(1u<<MT_WEEDS)|(1u<<MT_OCEAN))

/* --------------------------------------------------------------------- events ------- */
enum nm_event {       /* nmmo/lib/event_code.py [UPSTREAM]; members named at stat_wrapper.py:196-205,238-292 */
  EV_EAT_FOOD = 1, EV_DRINK_WATER = 2, EV_GO_FARTHEST = 3,
  EV_SCORE_HIT = 11, EV_PLAYER_KILL = 12,
  EV_CONSUME_ITEM = 21, EV_GIVE_ITEM = 22, EV_DESTROY_ITEM = 23, EV_HARVEST_ITEM = 24,
  EV_EQUIP_ITEM = 25, EV_LOOT_ITEM = 26,
  EV_GIVE_GOLD = 31, EV_LIST_ITEM = 32, EV_EARN_GOLD = 33, EV_BUY_ITEM = 34, EV_LOOT_GOLD = 35,
  EV_LEVEL_UP = 41
};
#define NM_N_EVENT 17   /* dense event index 0..16 in the order above */
/* unique-event key space: (dense event, type 0..17, level 0..10) -> bit index */
#define NM_UNIQ_LEVELS 11
#define NM_UNIQ_BITS (NM_N_EVENT * IT_N * NM_UNIQ_LEVELS)    /* 3366 */
#define NM_UNIQ_WORDS 106                                     /* ceil(3366/32) */

enum nm_skill { SK_MELEE = 1, SK_RANGE, SK_MAGE, SK_FISHING, SK_HERBALISM, SK_PROSPECTING,
                SK_CARVING, SK_ALCHEMY };

/* -------------------------------------------------------------------- actions ------- */
/* flat MultiDiscrete(12) column order: takeru/policy.py:293-307 */
enum nm_action {
  AC_ATTACK_STYLE = 0, AC_ATTACK_TARGET, AC_BUY_ITEM, AC_DESTROY_ITEM, AC_GIVE_ITEM,
  AC_GIVE_TARGET, AC_GOLD_PRICE, AC_GOLD_TARGET, AC_MOVE_DIR, AC_SELL_ITEM, AC_SELL_PRICE,
  AC_USE_ITEM, AC_N = 12
};
/* Direction edges [UPSTREAM nmmo/core/action.py]: North, South, East, West, Stay */
#define NM_DIR_N 5

/* ---------------------------------------------------------- per-agent stat block ---- */
/* int32 accumulators folded from the event stream (stat_wrapper.py:216-288) */
enum nm_stat {
  ST_EVT0 = 0,                         /* 17 event counters (dense index) */
  ST_EQUIP_FLAGS = 17,                 /* bit0 armor bit1 weapon bit2 tool bit3 ammo, bit4 harvest_weapon */
  ST_MAX_PROGRESS, ST_EARNED_GOLD, ST_MAX_DAMAGE,
  ST_MAXLVL_ARMOR, ST_MAXLVL_WEAPON, ST_MAXLVL_TOOL, ST_MAXLVL_AMMO, ST_MAXLVL_CONSUMABLE, /* -1 = none */
  ST_AGENT_KILLS, ST_NPC_KILLS,
  ST_UNIQ_PREV, ST_UNIQ_CURR,          /* stat_wrapper.py:124-126 */
  ST_TASK_ACC0, ST_TASK_ACC1,          /* predicate accumulators */
  ST_REWARD_SIGNALS,                   /* Task.reward_signal_count */
  ST_TASK_DONE,                        /* Task.completed */
  ST_PREV_PRICE,                       /* start_kit/reward_wrapper.py:52,59 */
  ST_Y_HP, ST_Y_EXP, ST_Y_DMG_INFLICTED, ST_Y_GOLD,   /* yaofeng/reward_wrapper.py:53-63 previous-tick values */
  ST_N = 40
};
/* double accumulators per agent */
enum nm_dstat { DS_CUM_REWARD = 0, DS_PROGRESS, DS_MAX_PROGRESS, DS_N };

/* ------------------------------------------------------------ episode info record ---- */
/* float32 record written when an agent terminates or is truncated (stat_wrapper.py:132-185) */
enum nm_info {
  IN_LENGTH = 0, IN_RETURN,
  IN_COD_ATTACKED, IN_COD_STARVED, IN_COD_DEHYDRATED,
  IN_TASK_COMPLETED, IN_TASK_2_REWARD_SIGNAL, IN_TASK_0P2_MAX_PROGRESS,
  IN_CURR_MAX_PROGRESS, IN_CURR_REWARD_SIGNALS,
  IN_MAX_COMBAT_LEVEL, IN_MAX_HARVEST_AMMO, IN_MAX_HARVEST_CONSUM,
  IN_MAX_PROGRESS_TO_CENTER, IN_EARNED_GOLD, IN_MAX_DAMAGE,
  IN_MAXLVL_ARMOR, IN_MAXLVL_WEAPON, IN_MAXLVL_TOOL, IN_MAXLVL_AMMO, IN_MAXLVL_CONSUMABLE, /* NaN = key absent */
  IN_AGENT_KILLS, IN_NPC_KILLS, IN_UNIQUE_EVENTS,
  IN_EV_EAT_FOOD, IN_EV_DRINK_WATER, IN_EV_SCORE_HIT, IN_EV_PLAYER_KILL, IN_EV_CONSUME_ITEM,
  IN_EV_HARVEST_ITEM, IN_EV_LIST_ITEM, IN_EV_BUY_ITEM,
  IN_EQUIP_ARMOR, IN_EQUIP_WEAPON, IN_EQUIP_TOOL, IN_EQUIP_AMMO, IN_HARVEST_WEAPON,
  IN_TASK_ID,
  IN_N = 40
};

/* ---------------------------------------------------------------------- tasks ------- */
/* Closed predicate vocabulary (nmmo/task/base_predicates.py [UPSTREAM]); the names are the
 * ones the reference imports: curriculum_generation/manual_curriculum.py:8-29,
 * neurips23_evaluation/heldout_evaluation_task.py:7-20, syllabus_wrapper.py:58-70.
 * A task row is int32[12]: {pred, p0, p1, p2, flags (nm_task_flag), pred2, q0, combine, q1, q2, wa, wb}.
 * combine = 0: pred alone; 1: pred * pred2 (manual_curriculum.py:201-202 `InventorySpaceGE * TickGE`);
 * 2: (wa/1000) * pred + (wb/1000) * pred2 (manual_curriculum.py:119-122 `0.3 * EquipItem + 0.7 * GainExperience`).
 * pred2 takes (q0, q1, q2) and must be a state predicate (no event accumulator, no window scan). */
enum nm_pred {
  TP_NONE = 0, TP_TICK_GE, TP_COUNT_EVENT, TP_CAN_SEE_TILE, TP_CAN_SEE_AGENT, TP_OCCUPY_TILE,
  TP_ATTAIN_SKILL, TP_GAIN_EXPERIENCE, TP_EQUIP_ITEM, TP_SCORE_HIT, TP_HOARD_GOLD, TP_EARN_GOLD,
  TP_SPEND_GOLD, TP_MAKE_PROFIT, TP_INVENTORY_SPACE_GE, TP_OWN_ITEM, TP_CONSUME_ITEM,
  TP_HARVEST_ITEM, TP_LIST_ITEM, TP_BUY_ITEM, TP_DEFEAT_ENTITY, TP_FULLY_ARMED, TP_STAY_ALIVE,
  TP_DISTANCE_TRAVELED, TP_ALL_DEAD, TP_ALL_MEMBERS_WITHIN_RANGE, TP_CAN_SEE_GROUP, TP_N
};
#define NM_TASK_COLS 12
/* task flags (row column 4, "p3"): who the subject is and how a target given by name is resolved
 * (reward_to="team" and the "left_team" / "right_team_leader" ... targets of manual_curriculum.py:158-162,
 * syllabus_wrapper.py:226-240) */
enum nm_task_flag {
  TF_TEAM = 1,              /* reward_to="team": the subject is the assignee's whole team, every member gets the reward */
  TF_RELATIVE_TARGET = 2    /* p0 = team offset relative to the assignee's team (-1 left, +1 right, 0 own):
                               CanSeeAgent -> that team's leader, CanSeeGroup / AllDead -> that team (AllDead p1 = 1: its leader) */
};

/* Pending next-episode values (nmmo_set_next_episodes): bits of an env's flags byte, one per field its next automatic
 * reset takes from the device buffers instead of deriving it */
enum nm_next { NM_NEXT_SEED = 1, NM_NEXT_MAP = 2, NM_NEXT_TASKS = 4 };

/* ------------------------------------------------------------------------ rng ------- */
/* Draw sites.  A draw is addressed by (env seed, tick, site, idx, k) so that a parallel
 * device step and a sequential CPU step consume the same values in any order; recorded
 * draws are injected by the same key (nmmo_inject_rng). */
enum nm_site {
  RS_SPAWN_PERM = 1,     /* reset: Fisher-Yates over player spawn slots, idx = i */
  RS_RESILIENT,          /* reset: shuffle of resilient flags, idx = i */
  RS_NPC_DECIDE,         /* idx = entity row; k = draw ordinal inside decide() */
  RS_BUY_SHUFFLE,        /* idx = i of Fisher-Yates */
  RS_HARVEST,            /* idx = player row; k = skill id (weapon-drop roll) */
  RS_NPC_SPAWN,          /* idx = attempt; k = draw ordinal inside spawn() */
  RS_RESPAWN,            /* idx = tile index r*S+c */
  RS_MAP,                /* reset: map id draw */
  RS_TASK,               /* reset: task id draw, idx = player row */
  RS_ACTION,             /* uniform-valid action sampler (bench/tests): idx = player row, k = head */
  RS_N
};

/* ------------------------------------------------------------ observation record ---- */
/* One record per agent slot per tick.  Field order = sorted-key flatten of the nmmo obs dict
 * (ActionTargets{Attack{Style,Target},Buy,Destroy,Give{InventoryItem,Target},
 * GiveGold{Price,Target},Move,Sell{InventoryItem,Price},Use}, AgentId, CurrentTick, Entity,
 * Inventory, Market, Task, Tile) -- the order pufferlib's emulation flattens in and the one
 * agent_zoo/takeru/policy.py:293-307 documents for the action heads.  Native dtypes: masks
 * int8, ids/tables int16, Task fp16.  Every section starts 16-byte aligned and the record
 * stride is a multiple of 128 B so a warp stores it with full 16-byte vectors. */
typedef struct nm_obs_layout {
  int32_t n_ent, n_mkt, n_inv, n_price, task_dim, win;   /* win = 2*vision+1 */
  /* mask byte offsets inside the record */
  int32_t m_style, m_target, m_buy, m_destroy, m_give_item, m_give_target, m_gold_price,
          m_gold_target, m_move, m_sell_item, m_sell_price, m_use, m_end;
  int32_t o_ids;        /* int16 AgentId, int16 CurrentTick */
  int32_t o_entity;     /* int16 [n_ent][31] */
  int32_t o_inventory;  /* int16 [n_inv][16] */
  int32_t o_market;     /* int16 [n_mkt][16] */
  int32_t o_task;       /* fp16  [task_dim] */
  int32_t o_tile;       /* int16 [win*win][3] */
  int32_t stride;       /* bytes per record */
  int32_t alg_bytes;    /* unpadded payload bytes (roofline accounting) */
} nm_obs_layout;

static inline NM_HD int32_t nm_align16(int32_t x) { return (x + 15) & ~15; }

static inline NM_HD void nm_obs_layout_init(const int32_t *cfg, nm_obs_layout *L) {
  int32_t o = 0;
  L->n_ent = cfg[NC_N_ENT_OBS]; L->n_mkt = cfg[NC_N_MKT_OBS]; L->n_inv = cfg[NC_N_INV];
  L->n_price = cfg[NC_N_PRICE]; L->task_dim = cfg[NC_TASK_DIM]; L->win = 2 * cfg[NC_VISION] + 1;
  L->m_style = o;       o += 3;
  L->m_target = o;      o += L->n_ent + 1;
  L->m_buy = o;         o += L->n_mkt + 1;
  L->m_destroy = o;     o += L->n_inv + 1;
  L->m_give_item = o;   o += L->n_inv + 1;
  L->m_give_target = o; o += L->n_ent + 1;
  L->m_gold_price = o;  o += L->n_price;
  L->m_gold_target = o; o += L->n_ent + 1;
  L->m_move = o;        o += NM_DIR_N;
  L->m_sell_item = o;   o += L->n_inv + 1;
  L->m_sell_price = o;  o += L->n_price;
  L->m_use = o;         o += L->n_inv + 1;
  L->m_end = o;
  L->alg_bytes = o;
  o = nm_align16(o);
  L->o_ids = o;         o += 4;                          L->alg_bytes += 4;  o = nm_align16(o);
  L->o_entity = o;      o += L->n_ent * EA_N_OBS * 2;    L->alg_bytes += L->n_ent * EA_N_OBS * 2; o = nm_align16(o);
  L->o_inventory = o;   o += L->n_inv * IA_N_OBS * 2;    L->alg_bytes += L->n_inv * IA_N_OBS * 2; o = nm_align16(o);
  L->o_market = o;      o += L->n_mkt * IA_N_OBS * 2;    L->alg_bytes += L->n_mkt * IA_N_OBS * 2; o = nm_align16(o);
  L->o_task = o;        o += L->task_dim * 2;            L->alg_bytes += L->task_dim * 2;         o = nm_align16(o);
  L->o_tile = o;        o += L->win * L->win * 3 * 2;    L->alg_bytes += L->win * L->win * 3 * 2;
  L->stride = (o + 127) & ~127;
}

/* rng key packing for injected draws: tick 20b | site 4b | idx 24b | k 8b */
static inline NM_HD uint64_t nm_rng_key(uint32_t tick, uint32_t site, uint32_t idx, uint32_t k) {
  return ((uint64_t)(tick & 0xFFFFFu) << 36) | ((uint64_t)(site & 0xFu) << 32) |
         ((uint64_t)(idx & 0xFFFFFFu) << 8) | (uint64_t)(k & 0xFFu);
}

#ifdef __cplusplus
}
#endif
#endif /* NMMO_SPEC_H */
