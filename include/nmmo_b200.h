/*
 * nmmo_b200.h -- C ABI of the B200-native batched Neural MMO simulator.
 *
 * Drop-in boundary.  The reference drives its environments through the pufferlib
 * vectorisation object (`recv/send/async_reset/close`,
 * /root/reference/reinforcement_learning/clean_pufferl.py:106-118,175,293,357,563) that wraps
 * `nmmo.Env -> RewardWrapper -> PettingZooPufferEnv`
 * (/root/reference/reinforcement_learning/environment.py:55-74).  The reference has no FFI of
 * its own (100 % Python), so these entry points are what a ctypes binding for that seam binds;
 * nmmo_b200/vecenv.py is that binding and INTEGRATION.md shows the reference-side stub.
 *
 * Conventions: plain pointers and sizes only; every call returns 0 on success or a negative
 * nm_status code, with a message in nmmo_last_error(); no exceptions cross the ABI.  All device
 * buffers are owned by the handle and stay valid until nmmo_destroy; the *_ptr accessors return
 * device pointers (wrap them zero-copy, e.g. __cuda_array_interface__ / DLPack).  One handle per
 * GPU; calls on a handle are serialised by the caller; `stream` is a cudaStream_t (NULL = the
 * legacy default stream).  There is no CPU fallback: creating a handle without a CUDA device
 * fails with NM_ERR_CUDA.
 */
#ifndef NMMO_B200_H
#define NMMO_B200_H

#include <stdint.h>
#include "nmmo_spec.h"

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nmmo_handle nmmo_handle;

enum nm_err { NM_OK = 0, NM_ERR_ARG = -1, NM_ERR_CUDA = -2, NM_ERR_LIMIT = -3, NM_ERR_STATE = -4 };

/* Replaces: the vectorization constructor building `num_envs` x env_creator()
 * (clean_pufferl.py:106-114; environment.py:57-58 `nmmo.Env(Config(env))`, RewardWrapper kwargs).
 * cfg / fcfg: the vectors of nmmo_spec.h (built by nmmo_b200/config.py from the same
 * env / reward_wrapper namespaces).  maps: uint8 [n_maps][S][S] host memory (the reference loads
 * them from PATH_MAPS, environment.py:41).  tasks / task_embed: the curriculum
 * (environment.py:49) as int32 [n_tasks][NM_TASK_COLS] predicate rows (nmmo_spec.h: 12 columns) + fp16 [n_tasks][task_dim].
 * env_base: global index of this handle's env 0 (env sharding across GPUs).
 * NM_ERR_LIMIT, before anything is allocated on the device, for a record layout the kernels cannot write:
 * N_ENT_OBS outside 1..255, N_INV outside 1..16, N_MKT_OBS or N_PRICE < 1, the twelve ActionTargets heads
 * together > 1024 entries, TASK_DIM not a positive multiple of 8, or VISION outside 0..MAP_BORDER-1 (tile windows are
 * read unclamped, and the far side of the spawn ring is MAP_BORDER tiles from the map edge). */
int nmmo_create(const int32_t *cfg, int n_cfg, const double *fcfg, int n_fcfg, int n_envs, int device,
                int env_base, const uint8_t *maps, int n_maps, const int32_t *tasks,
                const uint16_t *task_embed, int n_tasks, nmmo_handle **out);

/* Replaces: vectorization.close() (clean_pufferl.py:563). */
int nmmo_destroy(nmmo_handle *h);

/* Replaces: vectorization.async_reset(seed) -> BaseStatWrapper.reset -> nmmo.Env.reset
 * (clean_pufferl.py:175; stat_wrapper.py:48-55).  seeds: host uint64 [E].  map_ids (host int32 [E])
 * and task_ids (host int32 [E][P]) may be NULL: then they are drawn from the env seed like
 * Env.reset draws map_id, and like the curriculum sampler assigns tasks.  env_mask (host uint8
 * [E], NULL = all) selects which envs reset.  Observations/masks of the reset envs are written. */
int nmmo_reset(nmmo_handle *h, const uint64_t *seeds, const int32_t *map_ids, const int32_t *task_ids,
               const uint8_t *env_mask, void *stream);

/* Replaces: vectorization.send(actions) + the worker-side step + recv()
 * (clean_pufferl.py:293,357; stat_wrapper.py:57-97; nmmo.Env.step).  actions: DEVICE int32
 * [E][P][12], column order of nmmo_spec.h nm_action (agent_zoo/takeru/policy.py:293-307).  Envs whose
 * episode ended on the previous call are reset instead of stepped (pufferlib semantics).
 * Launches 2 kernels on `stream`; results are in the buffers returned by the accessors. */
int nmmo_step(nmmo_handle *h, const int32_t *actions_dev, void *stream);

/* Replaces: send(actions) of one batch of an env pool (clean_pufferl.py:357 with envs_per_batch < num_envs): steps
 * envs [env_lo, env_hi) only.  actions: DEVICE int32 [env_hi - env_lo][P][12], row 0 = env env_lo, 16-byte aligned.
 * Launches the step and observation kernels of the range on `stream`; envs of the range whose episode ended on their
 * previous step are reset instead of stepped, as in nmmo_step.  The built-in random policy (nmmo_set_autosample) writes
 * the range's rows of its buffer.  Ranges on different streams may run at the same time when they do not overlap; calls
 * that touch the whole handle (nmmo_reset, nmmo_step) must be ordered after every range step in flight.
 * NM_ERR_ARG for an empty or out-of-bounds range or misaligned actions; NM_ERR_STATE while per-kernel timing or the
 * phase profiler is on (both describe whole-handle launches). */
int nmmo_step_envs(nmmo_handle *h, int env_lo, int env_hi, const int32_t *actions_dev, void *stream);

/* Same call with HOST buffers (the copy-in / copy-out path the reference pays today,
 * clean_pufferl.py:302-304,329): H2D of actions, step, D2H of reward/terminated/truncated/mask;
 * obs_out may be NULL (observations stay on the device for the policy) or a host buffer of
 * E*P*stride bytes.  Synchronises `stream` before returning. */
int nmmo_step_host(nmmo_handle *h, const int32_t *actions_host, float *rew_out, uint8_t *term_out,
                   uint8_t *trunc_out, uint8_t *mask_out, uint8_t *obs_out, void *stream);
/* The same with int16 actions (every head is narrower than 32768 entries): half the bytes over the
 * host link, which is what bounds this call.  A caller whose policy runs on the GPU narrows there
 * (`actions.to(torch.int16).cpu()`) before the copy the reference makes at clean_pufferl.py:329. */
int nmmo_step_host_i16(nmmo_handle *h, const int16_t *actions_host, float *rew_out, uint8_t *term_out,
                       uint8_t *trunc_out, uint8_t *mask_out, uint8_t *obs_out, void *stream);

/* The same with one byte per head: byte k of an agent's 12 bytes = index of head k (all heads but one have
 * at most 256 entries: 3 styles, N_ent+1 targets, N_inv+1 items, 99 prices, 5 directions); the wide head,
 * Buy.MarketItem (head 2, N_mkt+1 entries), keeps bits 8.. of its index in bits 2..7 of byte 0, above the
 * two bits of Attack.Style.  A quarter of the int32 bytes over the host link.  An index outside its head
 * is a no-op for that head, as in the other variants.  NM_ERR_LIMIT if a head does not fit.
 * On handles of 1024 environments or more the actions are copied as two env ranges on an internal copy stream (ordered
 * after whatever is queued on `stream`) and the step kernel of the first range runs underneath the copy of the second;
 * pinned host memory keeps the copies asynchronous. */
int nmmo_step_host_u8(nmmo_handle *h, const uint8_t *actions_host, float *rew_out, uint8_t *term_out,
                      uint8_t *trunc_out, uint8_t *mask_out, uint8_t *obs_out, void *stream);

/* Uniform-random valid actions from the current ActionTargets masks (BASELINE.json config 2),
 * keyed (seed, global env, tick, agent, head); writes DEVICE int32 [E][P][12]. */
int nmmo_sample_actions(nmmo_handle *h, uint64_t seed, int32_t *actions_dev, void *stream);

/* Scripted survival policy for long benchmark runs (uniform-random agents starve within ~35 ticks): every agent walks
 * to the nearest water / foliage tile of its observation window when hungry, explores otherwise, never fights or
 * trades.  Reads only the observation records; writes DEVICE int32 [E][P][12].  NM_ERR_LIMIT for a tile window of more
 * than 256 tiles (VISION > 7). */
int nmmo_forage_actions(nmmo_handle *h, uint64_t seed, int32_t *actions_dev, void *stream);

/* Built-in random policy: with a non-NULL DEVICE buffer int32 [E][P][12], every reset/step also
 * writes uniform-random valid actions for the new observations into it (identical draws to
 * nmmo_sample_actions(seed)); NULL switches it off.  Rows of absent agents are zeroed once, when the
 * agent leaves: hand in a zero-initialised buffer (or enable it before a reset). */
int nmmo_set_autosample(nmmo_handle *h, uint64_t seed, int32_t *actions_dev_out);

/* Device pointers to the step outputs (valid until nmmo_destroy, rewritten by each step). */
void *nmmo_obs_ptr(nmmo_handle *h);          /* uint8 [E*P][stride]  flat observation records */
void *nmmo_reward_ptr(nmmo_handle *h);       /* float [E*P] */
void *nmmo_terminated_ptr(nmmo_handle *h);   /* uint8 [E*P] */
void *nmmo_truncated_ptr(nmmo_handle *h);    /* uint8 [E*P] */
void *nmmo_mask_ptr(nmmo_handle *h);         /* uint8 [E*P]  agent present in this step's output */
void *nmmo_info_ptr(nmmo_handle *h);         /* float [E*P][IN_N]  episode-end info records */
void *nmmo_info_valid_ptr(nmmo_handle *h);   /* uint8 [E*P] */
void *nmmo_episode_done_ptr(nmmo_handle *h); /* uint8 [E]    infos[..]["episode_done"], stat_wrapper.py:93-95 */
void *nmmo_task_id_ptr(nmmo_handle *h);      /* int32 [E*P]  task-table row of every agent slot (this episode) */
void *nmmo_task_embed_ptr(nmmo_handle *h);   /* fp16  [n_tasks][task_dim]  the task embeddings (the Task block of a record) */
int nmmo_obs_stride(nmmo_handle *h);
/* Names of the step and observation kernel instantiations the handle's next launch uses, as a profiler lists them.
 * nmmo_create chooses the family, the envs per CTA and the compile-time shape from the configuration; the name is the
 * generic instantiation while the phase profiler is on, or, for the step kernel, while draws are injected. */
const char *nmmo_step_kernel_name(nmmo_handle *h);
const char *nmmo_obs_kernel_name(nmmo_handle *h);
int nmmo_num_envs(nmmo_handle *h);
int nmmo_num_agents(nmmo_handle *h);

/* Recorded-RNG injection: draws of env `env` whose key (nm_rng_key) appears in `keys` (host,
 * any order) return the paired value instead of the counter hash.  Replaces the draws the
 * reference takes from its numpy Generator.  n = 0 clears. */
int nmmo_inject_rng(nmmo_handle *h, int env, const uint64_t *keys, const uint32_t *vals, int n);

/* Full state of one env for parity diffs: int16 ent[R][EA_N] (row-major), int16
 * items[CAP][IS_N], uint8 map[S*S]; also the tick, map id and error flags. */
int nmmo_snapshot(nmmo_handle *h, int env, int16_t *ent, int16_t *items, uint8_t *map, int32_t *scalars16);

/* Task state of one env's agents, what the reference reads from `env.agent_task_map[id][0]`
 * (stat_wrapper.py:155-159): task_id int32 [P], completed int32 [P] (tick of completion, 0 = not yet),
 * reward_signal_count int32 [P], max_progress float64 [P].  Any pointer may be NULL. */
int nmmo_task_state(nmmo_handle *h, int env, int32_t *task_id, int32_t *completed, int32_t *reward_signals,
                    double *max_progress);

/* Episode statistics of finished agents since the last clear: sums[IN_N], counts[IN_N] (means
 * are sums/counts, clean_pufferl.py:381-390), counters[8] = slot-steps, agent-steps (mask
 * sum), finished episodes, event-ring overflows, bytes moved by the observation kernel, rejected
 * next-episode entries (nmmo_set_next_episodes), 2 spare.  Plain sums so ranks can all-reduce them. */
int nmmo_stats(nmmo_handle *h, double *sums, double *counts, uint64_t *counters, int clear);

/* Device-side error state (synchronises): NM_ERR_STATE when an environment produced more events in one tick than its
 * event ring holds (events were dropped: statistics and event-driven task progress of that env are wrong) since the
 * counters were last cleared.  nmmo_step is asynchronous and cannot report it; the host-buffer calls do.  Also
 * NM_ERR_STATE when an automatic reset rejected an out-of-range pending next-episode entry (nmmo_set_next_episodes). */
int nmmo_check(nmmo_handle *h);

/* Environment state (DESIGN.md 2.3): one fixed-size blob per env, `bytes` long (header included, a multiple of 128), that
 * holds everything a step reads and an earlier step or reset wrote: the tables, the agents' wrapper and task state, and
 * the outputs recv() returns.  A blob loads into any slot of any handle created from the same config, maps, task table
 * and task embeddings (a digest of them is in the header) and of the same kernel family; E, env_base, envs per CTA and
 * the std / generic kernel choice do not matter.  The loaded env continues exactly as the saved one would have: every
 * engine draw is keyed by the env's own seed.  The built-in random policy (nmmo_set_autosample, nmmo_sample_actions) is
 * keyed by the global slot, so its draws after a load are those of the destination slot. */
int nmmo_state_bytes(nmmo_handle *h, size_t *bytes);
/* Writes the blobs of envs env_ids[0..n) (HOST int32, duplicates allowed) to DEVICE uint8 [n][bytes] (16-byte aligned).
 * Asynchronous on `stream`.  NM_ERR_ARG for n < 1, an id out of range or misaligned states. */
int nmmo_save_envs(nmmo_handle *h, const int32_t *env_ids, int n, uint8_t *states_dev, void *stream);
/* Loads blob i of DEVICE uint8 [n][bytes] into env env_ids[i] (HOST int32, no duplicates; one blob may be repeated to
 * load it into several slots), then rewrites the observation records, ActionTargets masks and built-in-policy rows of
 * envs [min id, max id + 1) with the observation kernel, as nmmo_reset does: the loaded envs' become exactly those of
 * the tick they were saved at.  Synchronises `stream` and reads the headers back before it touches any device state;
 * the load and observation kernels then run on `stream`.  Like nmmo_reset it must be ordered after every range step in
 * flight.  Leaves the nmmo_stats sums and counters 0-2 alone.  NM_ERR_ARG (the handle is unchanged) for n < 1, an id
 * out of range, a duplicate id, misaligned states, a bad magic or format version, a blob of the other family, or a
 * digest mismatch; NM_ERR_STATE while per-kernel timing or the phase profiler is on. */
int nmmo_load_envs(nmmo_handle *h, const int32_t *env_ids, int n, const uint8_t *states_dev, void *stream);

/* Event log (DESIGN.md 2.4): the player events each env emitted in its last step, as the reference's event log holds
 * them.  enable = 1 allocates the staging (E * ring size * 8 bytes: 32 MB for 4096 envs of the default shape) and zeroes
 * every env's count (also when already on); 0 frees it.  From then on every step call (nmmo_step, nmmo_step_envs, the
 * step_host calls) keeps each stepped env's events; an env the call resets has none, and so has an env that nmmo_reset
 * resets or nmmo_load_envs loads (the events are not part of a state blob).  Synchronises the device, so it is ordered
 * after every range step in flight.  With the log off, the step kernels do what they did without it. */
int nmmo_set_event_log(nmmo_handle *h, int enable);
/* Rows of the events of envs [env_lo, env_hi) -> DEVICE int32 rows_dev[cap][9], each
 * [env, ent_id, tick, event, type, level, number, gold, target]: env is the handle's env index, ent_id the agent row + 1,
 * tick the env's tick after the step, event the reference's EventCode; number and gold are sign-extended, target is the
 * target's entity id (players > 0, NPCs < 0) for SCORE_HIT, PLAYER_KILL, LOOT_ITEM and LOOT_GOLD and 0 otherwise.
 * Columns 1..8 are those of the reference's EventLogger rows.  Order: env, then agent, then the order the agent's events
 * happened in.  DEVICE int32 count_dev[0] receives the number of rows of the range, which may exceed cap; rows beyond
 * cap are not written.  An env whose event ring overflowed has the events the ring kept (nmmo_check reports the
 * overflow).  Asynchronous on `stream`, no host synchronisation.  NM_ERR_STATE while the log is off; NM_ERR_ARG for an
 * empty, reversed or out-of-bounds range, cap < 0, or a NULL or not 4-byte-aligned pointer (rows_dev may be NULL when
 * cap = 0). */
int nmmo_events(nmmo_handle *h, int env_lo, int env_hi, int32_t *rows_dev, int cap, int32_t *count_dev, void *stream);

/* Pending next-episode values (DESIGN.md 2.5): what an env's next AUTOMATIC reset takes instead of deriving it, so that
 * a curriculum (in torch on the device, or on the host) steers every episode, not only the first.
 * enable = 1 allocates the buffers below (E * (13 + 4 * P) bytes) with every flag 0 (also when already on); 0 frees them.
 * Synchronises the device, so it is ordered after every range step in flight.  The accessors return NULL while off.
 *   flags  uint8  [E]     bits nm_next (nmmo_spec.h): NM_NEXT_SEED 1 | NM_NEXT_MAP 2 | NM_NEXT_TASKS 4
 *   seed   uint64 [E]     the next episode's env seed
 *   map    int32  [E]     its map id
 *   task   int32  [E][P]  its task-table rows, one per agent slot
 * When: only at an env's automatic reset inside a step call (nmmo_step, nmmo_step_envs, the nmmo_step_host calls: the
 * step after the one that ended its episode).  nmmo_reset and nmmo_load_envs neither use the values nor clear them.
 * What: a field is taken only when its bit is set; otherwise it is derived as without this feature: the seed is
 * nm_mix64(seed + 0x632BE59BD9B4E019) of the ending episode's seed, the map and the tasks are drawn from the new seed.
 * Consumption: the reset sets the env's flags byte to 0 and leaves the value arrays as they are, so a curriculum finds
 * the envs that need a new entry by flags == 0, on the device.  Teams (NC_TEAM_SIZE > 1): agent p takes the entry of its
 * team leader, the row the task draw is keyed by, so a team's tasks are uniform.  Out of range: a map id outside
 * [0, n_maps) or a team's task row outside [0, n_tasks) is never read through; that field (that team's task) is drawn as
 * if unset, counters[5] of nmmo_stats counts it and nmmo_check returns NM_ERR_STATE.  The values belong to the slot: they
 * are not part of a state blob.  Writes by the caller must be ordered before the step call that should see them and
 * after the one that last cleared the flags (e.g. on the stream the env is stepped on). */
int nmmo_set_next_episodes(nmmo_handle *h, int enable);
void *nmmo_next_flags_ptr(nmmo_handle *h);
void *nmmo_next_seed_ptr(nmmo_handle *h);
void *nmmo_next_map_ptr(nmmo_handle *h);
void *nmmo_next_task_ptr(nmmo_handle *h);

/* Per-kernel device timing (CUDA events recorded on the launching stream around the step kernel
 * and the observation kernel): enable, run steps, read the mean milliseconds per launch. */
int nmmo_timing(nmmo_handle *h, int enable);
int nmmo_timing_read(nmmo_handle *h, double *step_ms, double *obs_ms, int *n_launches);

/* Observation writer mode: 0 (default) stores only the bytes of each record that can differ from
 * what HBM already holds (records persist across ticks); 1 rewrites all bytes of all records. */
int nmmo_set_obs_full(nmmo_handle *h, int full);

/* Development aid: per-phase SM-clock profiles (64 counters: 0..31 step kernel, 32..63 observation kernel). */
int nmmo_profile(nmmo_handle *h, int enable, unsigned long long *out64);

const char *nmmo_last_error(void);

/* ------------------------------------------------------------------ rollout storage + GAE ----
 * Device-resident replacement of the trainer-side rollout arrays (SURVEY.md 8(f) rank 1).
 * Replaces: clean_pufferl.py:183-197 (the batch_size + 1 row arrays), :329-346 (masked append of
 * one recv() and `sort_keys.extend((env_id, step))`), :413-414 (sort by (env_id, step)) and
 * :424-436 (the GAE loop).  All data pointers are DEVICE pointers; nothing is copied to the host. */
typedef struct nmmo_rollout nmmo_rollout;
enum nm_rollout_buffer {     /* nmmo_rollout_buffer(which): rows = batch_size + 1 */
  NM_RB_OBS = 0,             /* uint8 [rows][obs_stride] */
  NM_RB_ACTIONS,             /* int32 [rows][12] */
  NM_RB_LOGPROBS, NM_RB_REWARDS, NM_RB_DONES, NM_RB_VALUES,   /* float32 [rows] */
  NM_RB_SLOT, NM_RB_STEP,    /* int32 [rows]: the sort key (env_id of the agent slot, step) */
  NM_RB_IDXS,                /* int32 [rows]: sample indices sorted by (slot, step)  (clean_pufferl.py:413) */
  NM_RB_ADVANTAGES,          /* float32 [rows]: advantages[t] for t < ptr - 1, in sorted order (:424-436) */
  /* compact mode only */
  NM_RB_MARKET,              /* uint8 [max_steps * n_envs][market_bytes]: the Market block of an env in a call, stored once, in call order */
  NM_RB_MARKET_SLOT,         /* int32 [rows]: the row's Market block (blocks of earlier calls + env of the call; step_index * n_envs + env for whole-handle calls) */
  NM_RB_TASK_ID              /* int32 [rows]: the row's task id (its Task block is the embedding of that task) */
};
int nmmo_rollout_create(int device, int batch_size, int n_slots, int obs_stride, nmmo_rollout **out);
/* Compact storage: the Market block (identical for every agent of an env in a step, 12 KB of the 25 KB record) is stored
 * once per (step, env) and the Task block (the embedding of the agent's task, 4 KB) as the task id; a row keeps the other
 * 9 KB.  NM_RB_OBS is then uint8 [rows][obs_stride - market_bytes - task_bytes]; nmmo_rollout_expand re-assembles whole
 * records, bit-identical to what the plain mode stores.  market_off / task_off: byte offsets of the sections in a record
 * (nm_obs_layout o_market / o_task); ids_off: offset of the int16 AgentId (o_ids; a record with AgentId 0 is the all-zero
 * record of an agent that died this tick and expands to zeros); max_steps: store calls between two resets. */
int nmmo_rollout_create_compact(int device, int batch_size, int n_slots, int obs_stride, int agents_per_env,
                                int market_off, int market_bytes, int task_off, int task_bytes, int ids_off, int max_steps,
                                nmmo_rollout **out);
/* task_id: DEVICE int32 [n_slots] (nmmo_task_id_ptr of the env handle). */
int nmmo_rollout_store_compact(nmmo_rollout *r, const uint8_t *obs, const int32_t *actions, const float *logprob,
                               const float *value, const float *reward, const float *done, const uint8_t *mask,
                               const uint8_t *learner_mask, const int32_t *task_id, int step, void *stream);
/* out[k] = full record of row idxs[k] (idxs NULL: row k), k < n; task_embed: DEVICE fp16 [n_tasks][task_dim]
 * (nmmo_task_embed_ptr); out: DEVICE uint8 [n][obs_stride].  The minibatch gather of clean_pufferl.py:439-443. */
int nmmo_rollout_expand(nmmo_rollout *r, const int32_t *idxs_dev, int n, const uint16_t *task_embed_dev, uint8_t *out_dev, void *stream);
int nmmo_rollout_destroy(nmmo_rollout *r);
/* ptr = 0, sort keys cleared (clean_pufferl.py:278, :414). */
int nmmo_rollout_reset(nmmo_rollout *r, void *stream);
/* Append the rows i of one step with mask[i] != 0 (and learner_mask[i] != 0 when given), in slot
 * order, up to the capacity (`indices = where(...)[: batch_size - ptr + 1]`, clean_pufferl.py:333-348).
 * obs uint8 [n_slots][obs_stride], actions int32 [n_slots][12], logprob/value/reward/done float32 [n_slots],
 * masks uint8 [n_slots]; `step` is the loop counter of clean_pufferl.py:281. */
int nmmo_rollout_store(nmmo_rollout *r, const uint8_t *obs, const int32_t *actions, const float *logprob,
                       const float *value, const float *reward, const float *done, const uint8_t *mask,
                       const uint8_t *learner_mask, int step, void *stream);
/* The same for the slots [slot_lo, slot_lo + n) of one call, e.g. one batch of an env pool: every argument covers
 * the call's n slots (obs uint8 [n][obs_stride], ...), the sort key is slot_lo + i and the running counts are kept per
 * global slot, so calls over different ranges sort and chain like one call over all slots.  task_id: NULL for a plain
 * rollout, DEVICE int32 [n] for a compact one, whose range must cover whole envs; there the Market block is stored once
 * per (call, env of the call), up to max_steps * n_slots / agents_per_env blocks between two resets (NM_ERR_LIMIT when
 * full).  nmmo_rollout_store / _store_compact are this call with slot_lo = 0, n = n_slots. */
int nmmo_rollout_store_range(nmmo_rollout *r, int slot_lo, int n, const uint8_t *obs, const int32_t *actions,
                             const float *logprob, const float *value, const float *reward, const float *done,
                             const uint8_t *mask, const uint8_t *learner_mask, const int32_t *task_id, int step, void *stream);
/* Rows stored so far (synchronises `stream`). */
int nmmo_rollout_ptr(nmmo_rollout *r, void *stream, int *ptr_out);
/* Sorted order + advantages of the stored rows; float32 arithmetic of the reference in its order. */
int nmmo_rollout_gae(nmmo_rollout *r, double gamma, double gae_lambda, void *stream);
void *nmmo_rollout_buffer(nmmo_rollout *r, int which);
const char *nmmo_rollout_last_error(void);

#ifdef __cplusplus
}
#endif
#endif /* NMMO_B200_H */
