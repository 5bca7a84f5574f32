// nmmo_obs.cu -- observation + ActionTargets writer (the HBM-bound kernel of the step).
//
// Replaces, per agent and per tick, nmmo's Observation.to_gym()/_make_action_targets()
// [UPSTREAM nmmo/core/observation.py], the RewardWrapper.observation() mask edits
// (agent_zoo/takeru/reward_wrapper.py:25-37, agent_zoo/neurips23_start_kit/reward_wrapper.py:46-54,
// agent_zoo/yaofeng/reward_wrapper.py:65-83)
// and pufferlib's flatten + pad of the nested observation (reinforcement_learning/environment.py:73),
// writing the flat record the policy reads on-device (agent_zoo/takeru/policy.py:39-64).
//
// Small family (nmmo_obs_kernel): one 512-thread CTA per environment, two CTAs per SM.  The entity table (31 observed
// columns + status), the live prefix of the item table and the 4-bit tile map are staged into shared memory with
// TMA bulk copies; the env-global Market block is built once in shared memory; the agents that need a record
// are compacted into a work list; a pre-pass with four threads per agent finds each agent's visible rows (in table
// order) and target bits; each warp then assembles whole agent records -- the ActionTargets masks as one 32-entry word
// per lane -- and streams them out with 16-byte st.global.cs stores, 512 contiguous bytes per warp instruction, the
// Market block of a record with one TMA bulk copy.  DESIGN.md section 4.2 has the measurements behind each choice.
// Big family (nmmo_obs_big_kernel, up to 1024 agents per env): NM_BIG_OBS_AGENTS agents per CTA, several CTAs per
// environment; the tables are read where they live (row-major entity table: an observed row is the first 62 bytes
// of its table row), only the per-row position words, the Market block and the per-agent lists are in shared memory.
#include "nmmo_device.cuh"

namespace {

struct OSmall {
  static constexpr bool kStage = true;
  static constexpr bool kStd = false;
  typedef StdShape Shape;
  // staged columns are 16 bytes apart from a multiple of 128: the four lanes that read columns c, c+1, c+2, c+3 of one row
  // (Entity gather) hit four different banks
  static __device__ __forceinline__ int ent_idx(int col, int row, int R) { return col * (R + NM_OBS_ENT_SKEW) + row; }
};
struct OStd : OSmall {
  static constexpr bool kStd = true;
};
struct OBig {
  static constexpr bool kStage = false;
  static constexpr bool kStd = false;
  typedef StdShape5 Shape;
  static __device__ __forceinline__ int ent_idx(int col, int row, int) { return row * NM_BIG_ENT_STRIDE + col; }
};

struct OCtx {
  const NmParams *p;
  const int32_t *c;
  int R, S, CAP, ICAP, P, NINV;
  const int16_t *ent;      // [31][R]
  const int16_t *status;   // [R]
  const int16_t *item;     // [IS_N][ICAP] staged prefix of the item table
  const int16_t *gitem;    // [IS_N][CAP] the table in HBM (rows >= ICAP)
  const uint32_t *map;
};
#define OENT(col, row) o.ent[V::ent_idx((col), (row), o.R)]
#define OITM(col, row) ((row) < o.ICAP ? o.item[(col) * o.ICAP + (row)] : o.gitem[(size_t)(col) * o.CAP + (row)])

template <class V>
__device__ __forceinline__ int o_use_level(const OCtx &o, int row, int type) {
  switch (type) {
    case IT_SPEAR: case IT_WHETSTONE: return OENT(EA_MELEE_LEVEL, row);
    case IT_BOW: case IT_ARROW: return OENT(EA_RANGE_LEVEL, row);
    case IT_WAND: case IT_RUNES: return OENT(EA_MAGE_LEVEL, row);
    case IT_ROD: return OENT(EA_FISHING_LEVEL, row);
    case IT_GLOVES: return OENT(EA_HERBALISM_LEVEL, row);
    case IT_PICKAXE: return OENT(EA_PROSPECTING_LEVEL, row);
    case IT_AXE: return OENT(EA_CARVING_LEVEL, row);
    case IT_CHISEL: return OENT(EA_ALCHEMY_LEVEL, row);
    default: {
      int l = 1;
      for (int col = EA_MELEE_LEVEL; col <= EA_ALCHEMY_LEVEL; col += 2) l = max(l, (int)OENT(col, row));
      return l;
    }
  }
}
// position of the r-th (0-based) set bit of x (r < popc(x)): five popc steps instead of the software loop behind __fns
__device__ __forceinline__ int nth_set_bit(uint32_t x, int r) {
  int pos = 0, c;
  c = __popc(x & 0xffffu); if (r >= c) { r -= c; pos += 16; x >>= 16; }
  c = __popc(x & 0xffu);   if (r >= c) { r -= c; pos += 8;  x >>= 8; }
  c = __popc(x & 0xfu);    if (r >= c) { r -= c; pos += 4;  x >>= 4; }
  c = __popc(x & 0x3u);    if (r >= c) { r -= c; pos += 2;  x >>= 2; }
  return pos + ((r >= (int)(x & 1u)) ? 1 : 0);
}
__device__ __forceinline__ void st16(uint8_t *dst, uint4 v) { __stcs((uint4 *)dst, v); }
__device__ __forceinline__ uint32_t pack2(int a, int b) { return (uint32_t)(uint16_t)a | ((uint32_t)(uint16_t)b << 16); }

}  // namespace

struct OBigStd : OBig {
  static constexpr bool kStd = true;
};

template <class V>
__device__ __forceinline__ void obs_body(const NmParams &prm) {
  extern __shared__ __align__(128) uint8_t smem[];
  constexpr int T = NM_OBS_THREADS, NW = T >> 5;      // (compile-time: the shared-memory map of the std kernels folds into immediates)
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // small: one CTA per env, all of its agents; big: AP agents per CTA, parts CTAs per env
  const NmCfg<V::kStd> c{prm.cfg};
  // record layout and table shape: immediates in the std instantiation, run-time values otherwise
  typedef typename V::Shape SH;
  constexpr nm_obs_layout kStdL = nm_std_layout();
  const nm_obs_layout &L = V::kStd ? kStdL : prm.L;
  const int P = V::kStd ? SH::P : prm.P, R = V::kStd ? SH::R : prm.R, S = V::kStd ? SH::S : prm.S;
  const int CAP = V::kStd ? SH::CAP : prm.CAP;
  const int ICAP = !V::kStage ? 0 : (V::kStd ? SH::ICAP : prm.ICAP);      // big family: no staged item prefix, every row is read in place
  const int NINV = V::kStd ? SH::NINV : c[NC_N_INV], vis = V::kStd ? SH::VIS : c[NC_VISION];
  const int AP = V::kStage ? P : min(P, NM_BIG_OBS_AGENTS);
  const int parts = V::kStage ? 1 : (P + AP - 1) / AP;
  // small family: highest env of [env_lo, env_hi) first -- the tables the step kernel wrote last are still in L2, and the
  // records this kernel writes last are the ones the next step kernel (lowest env first) reads first
  const int env = V::kStage ? prm.env_hi - 1 - (int)blockIdx.x : prm.env_lo + (int)blockIdx.x / parts;
  const int p_lo = V::kStage ? 0 : ((int)blockIdx.x % parts) * AP, p_hi = min(P, p_lo + AP);
  const int tick = prm.scalars[(size_t)env * NM_SC_N + SC_TICK];

  size_t off = 0;
  auto carve = [&](size_t bytes) { uint8_t *q = smem + off; off = (off + bytes + 15) & ~(size_t)15; return q; };
  const uint32_t ent_bytes = (uint32_t)(EA_N_OBS * R * 2), st_bytes = (uint32_t)(R * 2);
  const uint32_t ent_smem_bytes = (uint32_t)(EA_N_OBS * (R + NM_OBS_ENT_SKEW) * 2);
  const uint32_t item_bytes = (uint32_t)(IS_N * ICAP * 2), map_bytes = (uint32_t)(S * S / 2);
  const int16_t *const g_ent = prm.ent + (size_t)env * (V::kStage ? (size_t)EA_N * R : (size_t)NM_BIG_ENT_STRIDE * R);
  int16_t *s_ent = V::kStage ? (int16_t *)carve(ent_smem_bytes) : nullptr;
  int16_t *s_status = V::kStage ? (int16_t *)carve(st_bytes) : nullptr;
  int16_t *s_item = V::kStage ? (int16_t *)carve(item_bytes) : nullptr;
  const uint32_t *s_map = V::kStage ? (const uint32_t *)carve(map_bytes)        // 4 bits per tile
                                    : (const uint32_t *)(prm.map + (size_t)env * map_bytes);
  auto tile = [&](int i) -> int { return (int)((s_map[i >> 3] >> ((i & 7) * 4)) & 15u); };
  auto status_of = [&](int r) -> int { return V::kStage ? (int)s_status[r] : (int)g_ent[V::ent_idx(EA_STATUS, r, R)]; };
  int16_t *s_mkt = (int16_t *)carve((size_t)L.n_mkt * IA_N_OBS * 2);
  uint16_t *s_mkt_rows = (uint16_t *)carve((size_t)L.n_mkt * 2);
  uint16_t *s_inv = (uint16_t *)carve((size_t)AP * NINV * 2);      // indexed by p - p_lo
  int *s_invn = (int *)carve((size_t)AP * 4);
  int *s_scan = (int *)carve(128 * 4);
  // ActionTargets masks are built as bits: lane w of the warp that assembles a record holds mask entries [32w, 32w+32)
  // in one register (nmmo_create rejects layouts with more than 1024 entries); they become bytes only in the store
  const int stage_bytes = nm_align16(L.m_end);
  uint16_t *s_vis_all = (uint16_t *)carve((size_t)NW * ((L.n_ent * 2 + 15) & ~15));
  // built-in policy: the mask words of the last NM_OBS_BATCH agents of each warp (row stride 33 words), the agents they
  // belong to, and the picks on their way out
  uint32_t *s_bb_all = (uint32_t *)carve((size_t)NW * NM_OBS_BATCH * 33 * 4);
  uint16_t *s_ba_all = (uint16_t *)carve((size_t)NW * NM_OBS_BATCH * 2);
  int16_t *s_pick_all = (int16_t *)carve((size_t)NW * NM_OBS_BATCH * AC_N * 2);
  // per warp: NM_OBS_EROWS Entity rows on their way out (small family only: the big family gathers straight from its table)
  int16_t *s_ebuf_all = V::kStage ? (int16_t *)carve((size_t)NW * NM_OBS_EROWS * 64) : nullptr;
  const int R32 = (R + 31) & ~31, RW = R32 >> 5;
  uint32_t *s_pos = (uint32_t *)carve((size_t)R32 * 4);     // (row+7)<<16 | (col+7) of alive rows, padded to whole warps
  // cell index for the vision-window search: alive rows bucketed by NM_OBS_CELL x NM_OBS_CELL-tile cell.  A window
  // (2 * vision + 1 <= NM_OBS_CELL + 1 tiles wide) overlaps at most 2 x 2 cells, so an agent looks at the handful of rows
  // listed there instead of at every row of the table.
  const int ncx = (S + NM_OBS_CELL - 1) / NM_OBS_CELL, n_cells = ncx * ncx;
  int *s_cend = (int *)carve((size_t)(n_cells + 1) * 4);    // per cell: count, then (after the fill) the end of its row list
  uint16_t *s_crow = (uint16_t *)carve((size_t)R32 * 2);    // rows grouped by cell
  uint32_t *s_vbm_all = (uint32_t *)carve((size_t)NW * RW * 4);      // per warp: bitmap of the rows inside the agent's window
  int *s_head = (int *)carve((3 * AC_N + 2) * 4);       // head offsets, lengths, work-list length and cursor, heads by length
  uint64_t *s_hash = (uint64_t *)carve((size_t)AP * 8);     // built-in policy: one 64-bit draw per agent, computed by one thread each
  uint32_t *s_meta = (uint32_t *)carve((size_t)AP * 4);
  // work list entries: agent (relative to p_lo) | dead << 10 | the agent's two candidate ranges of the cell-ordered row list
  // (begin A << 12 | count A << 24 | begin B << 36 | count B << 48)
  uint64_t *s_work = (uint64_t *)carve((size_t)AP * 8);
  // per agent (pre-pass, a quad of threads per agent): up to 32 visible rows in table order (+ their count in slot 32;
  // row stride 33 halfwords so that the quads of a warp hit different banks) and the Attack / Give target bits of those rows
  // (only where the pre-pass can run: at most 32 bitmap words per agent, and room for the bitmaps in the batch words)
  const bool pre_ok = RW <= 32 && (size_t)AP * RW * 4 <= (size_t)NW * NM_OBS_BATCH * 33 * 4;
  uint16_t *s_va = pre_ok ? (uint16_t *)carve((size_t)AP * 33 * 2) : nullptr;
  uint32_t *s_tg = pre_ok ? (uint32_t *)carve((size_t)AP * 3 * 4) : nullptr;
  uint64_t *bar = (uint64_t *)carve(16);

  long long t_prev = clock64();
  int ph = 32;
#define OPHASE() do { if (!V::kStd && prm.prof && tid == 0) { long long t_ = clock64(); atomicAdd(&prm.prof[ph], (unsigned long long)(t_ - t_prev)); t_prev = t_; } ph++; } while (0)
  // The table loads go out before anything else: 41 TMA bulk copies (an entity column each, status, map, the live prefix
  // of each item column), one per lane of warp 0 -- not one thread issuing them one after the other while the CTA waits.
  // Nobody else touches the mbarriers before the CTA barrier that follows the polling below.
  const int item_hi = prm.scalars[(size_t)env * NM_SC_N + SC_ITEM_HI];     // rows >= item_hi are free
  if (V::kStage && warp == 0) {
    if (lane == 0) {
      mbar_init(bar, 1); mbar_init(bar + 1, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      mbar_expect_tx(bar, ent_bytes + st_bytes + map_bytes);
    }
    __syncwarp();
    const int16_t *ge = g_ent;
    if (NM_OBS_ENT_SKEW == 0) { if (lane == 0) bulk_g2s(s_ent, ge, ent_bytes, bar); }
    else
      #pragma unroll 1
      for (int k = lane; k < EA_N_OBS; k += 32) bulk_g2s(s_ent + k * (R + NM_OBS_ENT_SKEW), ge + (size_t)k * R, (uint32_t)(R * 2), bar);
    if (lane == 31) bulk_g2s(s_status, ge + (size_t)EA_STATUS * R, st_bytes, bar);
    if (lane == 30) bulk_g2s((void *)s_map, prm.map + (size_t)env * map_bytes, map_bytes, bar);
    // (the item copies wait for item_hi, a load from HBM; the copies above do not)
    const uint32_t col_bytes = (uint32_t)min(item_hi, ICAP) * 2;       // only the live prefix of each item column
    if (lane == 0) mbar_expect_tx(bar + 1, col_bytes * IS_N);
    __syncwarp();
    if (col_bytes && lane < IS_N) bulk_g2s(s_item + lane * ICAP, prm.item + ((size_t)env * IS_N + lane) * CAP, col_bytes, bar + 1);
  } else if (V::kStage && warp == 1 && lane < 3) {
    // L2 prefetch for a CTA that starts a few microseconds from now (envs are taken highest first): this kernel writes
    // 1.7 GB through L2 while it reads 0.2 GB of tables, so a table fetched on demand waits behind the writes
    const int env_next = env - NM_OBS_PREFETCH_AHEAD;
    if (env_next >= prm.env_lo) {
      if (lane == 0) bulk_prefetch_l2(prm.ent + (size_t)env_next * EA_N * R, (uint32_t)(EA_N_OBS * R * 2));
      else if (lane == 1) bulk_prefetch_l2(prm.ent + (size_t)env_next * EA_N * R + (size_t)EA_STATUS * R, st_bytes);
      else bulk_prefetch_l2(prm.map + (size_t)env_next * map_bytes, map_bytes);
    }
  }
  if (tid < AC_N) {
    const int off[AC_N] = {L.m_style, L.m_target, L.m_buy, L.m_destroy, L.m_give_item, L.m_give_target,
                           L.m_gold_price, L.m_gold_target, L.m_move, L.m_sell_item, L.m_sell_price, L.m_use};
    const int len[AC_N] = {3, L.n_ent + 1, L.n_mkt + 1, L.n_inv + 1, L.n_inv + 1, L.n_ent + 1, L.n_price,
                           L.n_ent + 1, NM_DIR_N, L.n_inv + 1, L.n_price, L.n_inv + 1};
    // heads in the order the batched sampler walks them: longest first, so that the lanes of one pass have similar trip counts
    const int ord[AC_N] = {AC_BUY_ITEM, AC_ATTACK_TARGET, AC_GIVE_TARGET, AC_GOLD_TARGET, AC_GOLD_PRICE, AC_SELL_PRICE,
                           AC_DESTROY_ITEM, AC_GIVE_ITEM, AC_SELL_ITEM, AC_USE_ITEM, AC_MOVE_DIR, AC_ATTACK_STYLE};
    s_head[tid] = off[tid]; s_head[AC_N + tid] = len[tid]; s_head[2 * AC_N + 2 + tid] = ord[tid];
  }
  #pragma unroll 1
  for (int i = tid; i < p_hi - p_lo; i += T) { s_invn[i] = 0; s_meta[i] = prm.obs_meta[(size_t)env * P + p_lo + i]; }
  #pragma unroll 1
  for (int i = tid; i <= n_cells; i += T) s_cend[i] = 0;
  if (prm.sample_out)      // (the whole warp would otherwise compute the same hash for its agent, 128 times per CTA)
    #pragma unroll 1
    for (int i = tid; i < p_hi - p_lo; i += T)
      s_hash[i] = nm_hash64(prm.sample_seed + (uint64_t)(prm.env_base + env), (uint32_t)tick, RS_ACTION, (uint32_t)(p_lo + i), 0);
  if (V::kStage && warp == 0) {      // one warp polls (sixteen would spin in the issue slots the SM's other CTA is using) ...
    while (!mbar_try_wait(bar, 0)) {}
    while (!mbar_try_wait(bar + 1, 0)) {}
  }
  __syncthreads();
  if (V::kStage) {                   // ... and every thread then observes the completed phases itself (returns at once)
    while (!mbar_try_wait(bar, 0)) {}
    while (!mbar_try_wait(bar + 1, 0)) {}
  }
  OPHASE();      // 32 load

  OCtx o;
  o.p = &prm; o.c = prm.cfg; o.R = R; o.S = S; o.CAP = CAP; o.ICAP = ICAP; o.P = P; o.NINV = NINV;
  o.gitem = prm.item + (size_t)env * IS_N * CAP;
  o.ent = V::kStage ? s_ent : g_ent; o.status = s_status; o.item = s_item; o.map = s_map;
  const int wrapper = c[NC_WRAPPER];
  const bool no_give = (wrapper == NW_TAKERU || wrapper == NW_YAOFENG) && c[NC_DISABLE_GIVE];
  const bool no_danger = wrapper == NW_YAOFENG && c[NC_NO_DANGEROUS_NPC];      // yaofeng/reward_wrapper.py:78-81
  // Work list.  Alive agents (a full record each) and agents that died since their record was last
  // written (one zero fill) are compacted in id order by the last warp -- here, underneath the other warps' list-building
  // passes, not in a barrier interval of its own.
  if (warp == NW - 1) {
    int n = 0;
    #pragma unroll 1
    for (int base = p_lo; base < p_hi; base += 32) {
      int p = base + lane;
      uint32_t meta = p < p_hi ? s_meta[p - p_lo] : 0u;
      bool alive = p < p_hi && status_of(p) == ES_ALIVE;
      bool work = alive || (p < p_hi && ((meta & OM_NONZERO) || prm.obs_full));
      unsigned bm = __ballot_sync(0xffffffffu, work);
      if (work) s_work[n + __popc(bm & ((1u << lane) - 1))] = (uint64_t)((p - p_lo) | (alive ? 0 : 0x400));
      n += __popc(bm);
    }
    if (lane == 0) { s_head[2 * AC_N] = n; s_head[2 * AC_N + 1] = 0; }
  }
  // one word per table row for the vision-window scan: an empty row can never match
  const bool use_cells = 2 * vis + 1 <= NM_OBS_CELL + 1;      // else (huge vision radius): every row is scanned
  #pragma unroll 1
  for (int r = tid; r < R32; r += T) {
    const bool live = r < R && status_of(r) == ES_ALIVE;
    uint32_t pos = 0x7fff7fffu;
    if (live) {
      const int er = OENT(EA_ROW, r), ec = OENT(EA_COL, r);
      pos = ((uint32_t)(er + vis) << 16) | (uint32_t)(ec + vis);
      if (use_cells) atomicAdd(&s_cend[(er / NM_OBS_CELL) * ncx + ec / NM_OBS_CELL], 1);
    }
    s_pos[r] = pos;
  }
  // ---- inventory lists (row order) and the market list (row order, first n_mkt) -------
  const int K = (item_hi + T - 1) / T;      // consecutive rows per thread
  int my_listed = 0;
  for (int k = 0; k < K; k++) {
    int i = tid * K + k;
    if (i < item_hi && OITM(IS_TYPE, i) != 0) {
      int owner = OITM(IS_OWNER, i);
      if (owner > p_lo && owner <= p_hi) { int slot = atomicAdd(&s_invn[owner - 1 - p_lo], 1); if (slot < NINV) s_inv[(owner - 1 - p_lo) * NINV + slot] = (uint16_t)i; }
      if (OITM(IS_PRICE, i) > 0) my_listed++;
    }
  }
  // block exclusive scan of my_listed -- and, in the same two barriers, of the per-cell row counts (each thread owns
  // CK consecutive cells; the counts were completed before the barrier that precedes the item pass... no: they are
  // complete here because the item pass below them reads nothing of theirs and a barrier follows the s_pos pass)
  const int CK = (n_cells + T - 1) / T;
  int my_cells = 0;
  __syncthreads();                                   // cell counts complete
  #pragma unroll 1
  for (int k = 0; k < CK; k++) { const int ci = tid * CK + k; if (ci < n_cells) my_cells += s_cend[ci]; }
  int incl = my_listed, cincl = my_cells;
  for (int d = 1; d < 32; d <<= 1) {
    int v = __shfl_up_sync(0xffffffffu, incl, d), cv = __shfl_up_sync(0xffffffffu, cincl, d);
    if (lane >= d) { incl += v; cincl += cv; }
  }
  if (lane == 31) { s_scan[warp] = incl; s_scan[64 + warp] = cincl; }
  __syncthreads();
  if (warp == 0) {
    int v = lane < NW ? s_scan[lane] : 0, inc2 = v, cv = lane < NW ? s_scan[64 + lane] : 0, cinc2 = cv;
    for (int d = 1; d < 32; d <<= 1) {
      int u = __shfl_up_sync(0xffffffffu, inc2, d), cu = __shfl_up_sync(0xffffffffu, cinc2, d);
      if (lane >= d) { inc2 += u; cinc2 += cu; }
    }
    if (lane < NW) { s_scan[32 + lane] = inc2 - v; s_scan[96 + lane] = cinc2 - cv; }
    if (lane == NW - 1) s_scan[63] = inc2;
  }
  __syncthreads();
  {   // counts -> start offsets (the fill below advances each to the end of its cell's list)
    int run = s_scan[96 + warp] + cincl - my_cells;
    #pragma unroll 1
    for (int k = 0; k < CK; k++) { const int ci = tid * CK + k; if (ci < n_cells) { const int cnt = s_cend[ci]; s_cend[ci] = run; run += cnt; } }
  }
  OPHASE();      // 33 lists + scan
  const int n_mkt = min(s_scan[63], L.n_mkt);
  {
    int pos = s_scan[32 + warp] + incl - my_listed;
    for (int k = 0; k < K; k++) {
      int i = tid * K + k;
      if (i < item_hi && OITM(IS_TYPE, i) != 0 && OITM(IS_PRICE, i) > 0) { if (pos < L.n_mkt) s_mkt_rows[pos] = (uint16_t)i; pos++; }
    }
  }
  #pragma unroll 1
  for (int p = tid; p < p_hi - p_lo; p += T) {           // sort each inventory list by row (<= 12 entries)
    int n = min(s_invn[p], NINV);
    uint16_t *l = s_inv + p * NINV;
    for (int i = 1; i < n; i++) { uint16_t x = l[i]; int j = i - 1; while (j >= 0 && l[j] > x) { l[j + 1] = l[j]; j--; } l[j + 1] = x; }
  }
  __syncthreads();
  if (use_cells) {      // fill the per-cell row lists (each cell's cursor ends at the end of its list)
    #pragma unroll 1
    for (int r = tid; r < R; r += T) {
      const uint32_t pos = s_pos[r];
      if (pos == 0x7fff7fffu) continue;
      const int er = (int)(pos >> 16) - vis, ec = (int)(pos & 0xffffu) - vis;
      const int k = atomicAdd(&s_cend[(er / NM_OBS_CELL) * ncx + ec / NM_OBS_CELL], 1);
      s_crow[k] = (uint16_t)r;
    }
  }
  #pragma unroll 1
  for (int j = tid; j < n_mkt; j += T) {       // the Market block, identical for every agent of the env
    int16_t row[IA_N_OBS];                      // (rows past n_mkt are zeros and are written as such, not staged)
    int i = s_mkt_rows[j];
    item_obs_row(c, i, OITM(IS_TYPE, i), OITM(IS_LEVEL, i), OITM(IS_OWNER, i), OITM(IS_QUANTITY, i), OITM(IS_EQUIPPED, i), OITM(IS_PRICE, i), row);
    uint4 *dst = (uint4 *)(s_mkt + j * IA_N_OBS);
    dst[0] = make_uint4(pack2(row[0], row[1]), pack2(row[2], row[3]), pack2(row[4], row[5]), pack2(row[6], row[7]));
    dst[1] = make_uint4(pack2(row[8], row[9]), pack2(row[10], row[11]), pack2(row[12], row[13]), pack2(row[14], row[15]));
  }
  fence_async_smem();      // the block is later read by bulk copies (async proxy)
  __syncthreads();
  OPHASE();      // 34 market rows

  // ---- per-agent records: one warp per agent -------------------------------------------
  uint32_t *bb = s_bb_all + warp * (NM_OBS_BATCH * 33);
  uint16_t *ba = s_ba_all + warp * NM_OBS_BATCH;
  int16_t *picks = s_pick_all + warp * (NM_OBS_BATCH * AC_N);
  int16_t *ebuf = s_ebuf_all + warp * (NM_OBS_EROWS * 32);
  // the bits of mask entries [lo, hi) / of entry pos that fall into this lane's word
  auto range_bits = [&](int lo, int hi) -> uint32_t {
    const int a = max(lo - 32 * lane, 0), b = min(hi - 32 * lane, 32);
    if (b <= a) return 0u;
    return (b >= 32 ? 0xffffffffu : ((1u << b) - 1u)) & ~((1u << a) - 1u);
  };
  auto one_bit = [&](int pos) -> uint32_t { return (pos >> 5) == lane ? 1u << (pos & 31) : 0u; };
  // entries that do not depend on the agent (Style, Sell.Price, the no-op slots, GiveGold.Price[0])
  const uint32_t tmpl_word = range_bits(L.m_style, L.m_style + 3) | range_bits(L.m_sell_price, L.m_sell_price + L.n_price) |
                             one_bit(L.m_buy + L.n_mkt) | one_bit(L.m_destroy + L.n_inv) | one_bit(L.m_give_item + L.n_inv) |
                             one_bit(L.m_sell_item + L.n_inv) | one_bit(L.m_use + L.n_inv) | one_bit(L.m_give_target + L.n_ent) |
                             one_bit(L.m_gold_target + L.n_ent) | one_bit(L.m_gold_price);
  uint16_t *s_vis = s_vis_all + (size_t)warp * (((L.n_ent * 2 + 15) & ~15) / 2);
  const uint4 zero4 = make_uint4(0, 0, 0, 0);
  long long n_stored = 0;                     // 16-byte chunks stored by this warp
  // (the work list was compacted by the last warp right after the tables arrived)
  const int n_work = s_head[2 * AC_N];
  if (use_cells) {
    // Pre-pass, four threads per agent (the whole CTA for 128 agents).  The rows listed in the (at most 2 x 2) cells under
    // an agent's window are two contiguous ranges of the cell-ordered row list.  With at most 32 candidates (the common
    // case) the quad also finds the visible rows, puts them in table order and works out their target bits -- work that
    // keeps one lane in three busy when a whole warp does it for one agent.
    // (scratch: one row bitmap per agent, in the sampler's batch words, which are not in use yet; without room for them,
    //  or with more than 32 bitmap words per agent, every agent takes the warp path)
    uint32_t *s_pbm = s_bb_all;
    const int WPL = (RW + 3) >> 2;                    // bitmap words per lane of a quad
    #pragma unroll 1
    for (int wi0 = 0; wi0 < n_work; wi0 += T / 4) {
      const int wi = wi0 + (tid >> 2), q = lane & 3;
      const uint64_t e = wi < n_work ? s_work[wi] : (uint64_t)0x400;
      const bool alive = !((uint32_t)e & 0x400u);
      const int pa = (int)((uint32_t)e & 0x3ffu), p = p_lo + pa;
      int r0 = 0, c0 = 0, begA = 0, nA = 0, begB = 0, n_cand = 0;
      if (alive) {
        r0 = OENT(EA_ROW, p); c0 = OENT(EA_COL, p);
        const int cr0 = (int)((unsigned)max(r0 - vis, 0) / NM_OBS_CELL), cr1 = (int)((unsigned)min(r0 + vis, S - 1) / NM_OBS_CELL);
        const int cc0 = (int)((unsigned)max(c0 - vis, 0) / NM_OBS_CELL), cc1 = (int)((unsigned)min(c0 + vis, S - 1) / NM_OBS_CELL);
        const int ca = cr0 * ncx + cc0;
        begA = ca ? s_cend[ca - 1] : 0;
        const int endA = s_cend[cr0 * ncx + cc1];
        int endB = 0;
        if (cr1 > cr0) { const int cb = cr1 * ncx + cc0; begB = s_cend[cb - 1]; endB = s_cend[cr1 * ncx + cc1]; }
        nA = endA - begA; n_cand = nA + endB - begB;
        if (q == 0) s_work[wi] = e | ((uint64_t)begA << 12) | ((uint64_t)nA << 24) | ((uint64_t)begB << 36) | ((uint64_t)(endB - begB) << 48);
      }
      const bool fast = pre_ok && alive && n_cand <= 32;      // else the assembling warp searches (bitmap walk)
      uint32_t *bm = s_pbm + pa * RW;
      uint16_t *va = s_va + pa * 33;
      if (fast)
        #pragma unroll 1
        for (int t = 0; t < WPL; t++) if (q * WPL + t < RW) bm[q * WPL + t] = 0;
      __syncwarp();
      // candidates q, q + 4, ...: the hits are marked in the agent's row bitmap
      const int its = (__reduce_max_sync(0xffffffffu, fast ? n_cand : 0) + 3) >> 2;
      #pragma unroll 1
      for (int it = 0; it < its; it++) {
        const int i = it * 4 + q;
        if (fast && i < n_cand) {
          const int row = s_crow[i < nA ? begA + i : begB + i - nA];
          const uint32_t pos = s_pos[row];
          if ((uint32_t)((int)(pos >> 16) - r0) <= (uint32_t)(2 * vis) && (uint32_t)((int)(pos & 0xffffu) - c0) <= (uint32_t)(2 * vis))
            atomicOr(&bm[row >> 5], 1u << (row & 31));
        }
      }
      __syncwarp();
      // table order = bitmap order: a lane counts its words, the quad's prefix gives it its place, it writes its rows
      int cnt = 0;
      if (fast)
        #pragma unroll 1
        for (int t = 0; t < WPL; t++) if (q * WPL + t < RW) cnt += __popc(bm[q * WPL + t]);
      const int qb = lane & 28;
      const int c_0 = __shfl_sync(0xffffffffu, cnt, qb), c_1 = __shfl_sync(0xffffffffu, cnt, qb + 1);
      const int c_2 = __shfl_sync(0xffffffffu, cnt, qb + 2), c_3 = __shfl_sync(0xffffffffu, cnt, qb + 3);
      int idx = (q > 0 ? c_0 : 0) + (q > 1 ? c_1 : 0) + (q > 2 ? c_2 : 0);
      int nv = min(c_0 + c_1 + c_2 + c_3, L.n_ent);      // (at most 32: one hit per candidate)
      if (fast)
        #pragma unroll 1
        for (int t = 0; t < WPL; t++) {
          const int w = q * WPL + t;
          uint32_t bits = w < RW ? bm[w] : 0u;
          #pragma unroll 1
          while (bits && idx < nv) { const int b2 = __ffs(bits) - 1; bits &= bits - 1; va[idx++] = (uint16_t)(w * 32 + b2); }
        }
      if (pre_ok && alive && q == 0) va[32] = fast ? (uint16_t)nv : (uint16_t)0xffff;
      __syncwarp();
      uint32_t att = 0, give = 0, any = 0;
      if (fast) {
        const int my_id = OENT(EA_ID, p);
        const bool immune = OENT(EA_TIME_ALIVE, p) < c[NC_SPAWN_IMMUNITY], has_inv = s_invn[pa] > 0;
        #pragma unroll 1
        for (int i = q; i < nv; i += 4) {
          const int row = va[i], id = OENT(EA_ID, row), npc_type = OENT(EA_NPC_TYPE, row);
          const uint32_t pos = s_pos[row];
          const int er = (int)(pos >> 16) - vis, ec = (int)(pos & 0xffffu) - vis;
          const bool ok = nm_linf(er, ec, r0, c0) <= c[NC_REACH] && id != my_id && !(immune && id > 0);
          any |= ok;                                             // the no-op entry is the engine's, before the wrapper edit
          if (ok && !(no_danger && npc_type > 1)) att |= 1u << i;
          if (!no_give && has_inv && er == r0 && ec == c0 && npc_type == 0 && id != my_id) give |= 1u << i;
        }
      }
      att |= __shfl_xor_sync(0xffffffffu, att, 1); give |= __shfl_xor_sync(0xffffffffu, give, 1); any |= __shfl_xor_sync(0xffffffffu, any, 1);
      att |= __shfl_xor_sync(0xffffffffu, att, 2); give |= __shfl_xor_sync(0xffffffffu, give, 2); any |= __shfl_xor_sync(0xffffffffu, any, 2);
      if (fast && q == 0) { uint32_t *tg = s_tg + pa * 3; tg[0] = att; tg[1] = give; tg[2] = any; }
    }
    __syncthreads();
  }
  OPHASE();      // 35 work list
  // Tile window, fast path (window at least 8 wide, at most 32 groups of 8 tiles): lane g owns tiles 8g..8g+7 of
  // the row-major window, which lie in at most two window rows.  Where they lie does not depend on the agent.
  const int tw_tiles = L.win * L.win, tw_groups = (tw_tiles + 7) / 8;
  const bool tw_fast = L.win >= 8 && tw_groups <= 32;
  const int tw_dr = (lane * 8) / L.win, tw_dc = (lane * 8) - tw_dr * L.win;
  const int tw_first = min(8, L.win - tw_dc);             // tiles of the group in its first window row
  const int tw_nval = min(8, max(0, tw_tiles - lane * 8));                 // tiles of the group that exist
  const uint32_t tw_matmask = tw_nval >= 8 ? 0xffffffffu : ((1u << (4 * tw_nval)) - 1u);
  const uint32_t tw_full = tw_nval == 8 ? 0xffffffffu : 0u, tw_unit = tw_full & 0x10000u;      // a column step; 0 where tiles 1..7 do not exist
  auto fetch8 = [&](int i) -> uint32_t {                    // the 8 nibbles of tiles i..i+7
    const int w = i >> 3, sh = (i & 7) * 4;
    return __funnelshift_r(s_map[w], s_map[w + 1], sh);
  };
  long long w_t0 = clock64();
  // Work items are dealt round-robin when most agents are alive (items of equal cost: no queue traffic) and pulled from a
  // shared cursor otherwise (a zero fill is much cheaper than a record, so a static deal would leave warps idle)
  const bool deal = 2 * n_work > AP;
  const int its_dealt = deal ? (n_work / NW) * NM_OBS_DEAL_NUM / 8 : 0;      // (NM_OBS_DEAL_NUM eighths; the remainder is pulled)
  // obs_full = 1: every row of every section is rewritten, the Task block included
  const int ms_shift = (lane & 1) * 16;      // mask store: which half of the source word this lane expands
  const uint32_t meta_full = (uint32_t)L.n_ent | ((uint32_t)L.n_inv << 8) | ((uint32_t)L.n_mkt << 18);
  int nb = 0;                                 // agents whose mask words wait in bb for the built-in policy
  #pragma unroll 1
  for (int it = 0;; it++) {
    int wi = warp + it * NW;
    if (it >= its_dealt) {
      if (lane == 0) wi = its_dealt * NW + atomicAdd(&s_head[2 * AC_N + 1], 1);
      wi = __shfl_sync(0xffffffffu, wi, 0);
    }
    // ---- built-in random policy (optional): uniform over the valid entries of every head ----
    // Run for NM_OBS_BATCH agents at a time so that a lane resolves one (agent, head) pair and all lanes are busy:
    // count the head's set bits in the agent's mask words, draw, find the drawn entry.  Same draws as nmmo_sample_kernel.
    if (nb == NM_OBS_BATCH || (wi >= n_work && nb > 0)) {
      __syncwarp();
      const int n_items = nb * AC_N;
      // item / nb by multiplication (exact for item < 2^10, nb <= 2^6); a full batch needs no division at all
      const int rcp = nb == NM_OBS_BATCH ? (65536 + NM_OBS_BATCH - 1) / NM_OBS_BATCH : (65536 + nb - 1) / nb;
      #pragma unroll 1
      for (int i0 = 0; i0 < n_items; i0 += 32) {
        const int item = i0 + lane;
        if (item < n_items) {
          const int hi = (item * rcp) >> 16, sl = item - hi * nb;          // heads of similar length share a pass
          const int h = s_head[2 * AC_N + 2 + hi], o0 = s_head[h];
          int o1 = o0 + s_head[AC_N + h];
          const uint32_t *bits = bb + sl * 33;
          const uint64_t base64 = s_hash[ba[sl]];
          bool stay = false;
          if (h == AC_MOVE_DIR && c[NC_SAMPLE_MOVE_PCT] > 0) {
            // Move-biased workload (BASELINE.json configs[4]): with the given probability a valid direction other
            // than Stay (the head then covers the four directions only), else Stay
            const uint32_t four = __funnelshift_r(bits[o0 >> 5], bits[(o0 >> 5) + 1], o0 & 31) & 15u;
            if (four) { if (nm_bounded(nm_action_draw(base64, AC_N), 100) < c[NC_SAMPLE_MOVE_PCT]) o1 = o0 + 4; else stay = true; }
          }
          // only the non-zero words of the head's range are looked at (bits[32]: which of the agent's words are non-zero)
          const int w0 = o0 >> 5, w1 = (o1 - 1) >> 5;
          const uint32_t wm = bits[32] & (0xffffffffu << w0) & (0xffffffffu >> (31 - w1));
          const uint32_t lo_mask = 0xffffffffu << (o0 & 31), hi_mask = 0xffffffffu >> ((32 - o1) & 31);
          auto word_at = [&](int w) -> uint32_t {
            uint32_t x = bits[w];
            if (w == w0) x &= lo_mask;
            if (w == w1) x &= hi_mask;
            return x;
          };
          int pick = 0;
          if (stay) pick = 4;
          else {
            int total = 0;
            #pragma unroll 1
            for (uint32_t mm = wm; mm; mm &= mm - 1) total += __popc(word_at(__ffs(mm) - 1));
            if (total > 0) {
              int jj = nm_bounded(nm_action_draw(base64, h), total);
              int wsel = w1;
              #pragma unroll 1
              for (uint32_t mm = wm; mm; mm &= mm - 1) {
                const int w = __ffs(mm) - 1, cnt = __popc(word_at(w));
                if (jj < cnt) { wsel = w; break; }
                jj -= cnt;
              }
              pick = wsel * 32 + nth_set_bit(word_at(wsel), jj) - o0;
            }
          }
          picks[sl * AC_N + h] = (int16_t)pick;
        }
      }
      __syncwarp();
      #pragma unroll 1
      for (int i = lane; i < n_items; i += 32) {      // out in agent-major order: 48 contiguous bytes per agent
        const int sl = i / AC_N;
        prm.sample_out[((size_t)env * P + p_lo + ba[sl]) * AC_N + (i - sl * AC_N)] = picks[i];
      }
      __syncwarp();
      nb = 0;
    }
    if (wi >= n_work) break;
    const uint64_t went = s_work[wi];
    const int p = p_lo + (int)((uint32_t)went & 0x3ffu);
    const size_t a = (size_t)env * P + p;
    uint8_t *rec = prm.obs + a * L.stride;
    // The record lives in HBM across ticks, so only bytes that can differ from last tick's
    // record are stored.  meta remembers what the record currently holds: rows of Entity /
    // Inventory / Market that are non-zero, whether the Task block is in place, whether the
    // record is non-zero at all.  obs_full = 1 rewrites every byte (roofline / A-B mode).
    const uint32_t meta = s_meta[p - p_lo];
    if ((uint32_t)went & 0x400u) {           // dead or absent agents get the zero pad record
      // ... and every head of the built-in policy picks 0: written once, when the agent leaves (the action
      // buffer must start zeroed, which nmmo_set_autosample's caller guarantees)
      if (prm.sample_out && lane < AC_N) prm.sample_out[a * AC_N + lane] = 0;
      for (int k = lane; k < L.stride / 16; k += 32) st16(rec + k * 16, zero4);
      n_stored += L.stride / 16;
      if (lane == 0) s_meta[p - p_lo] = 0;
      continue;
    }
    const uint32_t held = prm.obs_full ? meta_full : meta;      // what the record is taken to hold
    const int pv = (int)(held & 255u), pi = (int)((held >> 8) & 31u), pm = (int)((held >> 18) & 1023u);
    const bool task_ok = (held & OM_TASK) != 0;
    const int r0 = OENT(EA_ROW, p), c0 = OENT(EA_COL, p), my_id = OENT(EA_ID, p), my_gold = OENT(EA_GOLD, p);
    // visible entities: table rows inside the window, in table order, first n_ent
    int n_vis = 0;
    // |r - r0| <= vis  <=>  0 <= (r + vis) - r0 <= 2*vis, same for the column
    auto in_window = [&](uint32_t pos) -> bool {
      return (uint32_t)((int)(pos >> 16) - r0) <= (uint32_t)(2 * vis) && (uint32_t)((int)(pos & 0xffffu) - c0) <= (uint32_t)(2 * vis);
    };
    // candidates: the agent's two ranges of the cell-ordered row list (found when the work list was built)
    const int begA = (int)((uint32_t)(went >> 12) & 0xfffu), nA = (int)((uint32_t)(went >> 24) & 0xfffu);
    const int begB = (int)((uint32_t)(went >> 36) & 0xfffu), nB = (int)((uint32_t)(went >> 48) & 0xfffu);
    const int n_cand = nA + nB;
    // the common case (at most 32 candidates): the list and the target bits were made by the pre-pass
    const uint16_t *vl = s_va + (p - p_lo) * 33;      // this agent's visible rows, in table order
    const bool pre = use_cells && pre_ok && vl[32] != 0xffffu;
    if (pre) {
      n_vis = vl[32];
    } else if (use_cells) {
      // many candidates: they are tested and marked in a row bitmap; walking the bitmap yields them in table order
      uint32_t *vbm = s_vbm_all + warp * RW;
      #pragma unroll 1
      for (int w = lane; w < RW; w += 32) vbm[w] = 0;
      __syncwarp();
      #pragma unroll 1
      for (int i = lane; i < n_cand; i += 32) {
        const int row = s_crow[i < nA ? begA + i : begB + i - nA];
        if (in_window(s_pos[row])) atomicOr(&vbm[row >> 5], 1u << (row & 31));
      }
      __syncwarp();
      #pragma unroll 1
      for (int w0 = 0; w0 < RW; w0 += 32) {
        const int w = w0 + lane;
        uint32_t bits = w < RW ? vbm[w] : 0u;
        const int pc = __popc(bits);
        if (!__any_sync(0xffffffffu, pc)) continue;
        int incl2 = pc;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(0xffffffffu, incl2, d); if (lane >= d) incl2 += u; }
        int idx = n_vis + incl2 - pc;
        #pragma unroll 1
        while (bits && idx < L.n_ent) { const int b = __ffs(bits) - 1; bits &= bits - 1; s_vis[idx++] = (uint16_t)(w * 32 + b); }
        n_vis += __shfl_sync(0xffffffffu, incl2, 31);
      }
    } else {
      #pragma unroll 1
      for (int base = 0; base < R; base += 32) {
        int row = base + lane;
        const bool in = in_window(s_pos[row]);               // padded: rows >= R hold the never-matching word
        unsigned bm = __ballot_sync(0xffffffffu, in);
        if (!bm) continue;
        if (in) { int idx = n_vis + __popc(bm & ((1u << lane) - 1)); if (idx < L.n_ent) s_vis[idx] = (uint16_t)row; }
        n_vis += __popc(bm);
      }
    }
    n_vis = min(n_vis, L.n_ent);
    const int n_inv = min(s_invn[p - p_lo], NINV);
    const uint16_t *inv = s_inv + (p - p_lo) * NINV;
    if (!pre) vl = s_vis;
    __syncwarp();      // s_vis is complete
    // ---- ActionTargets (as bits: this lane's word of the record's mask entries) ----
    uint32_t mw = tmpl_word;
    // a ballot over up to 32 consecutive entries, the first of them entry o of the masks
    auto place = [&](uint32_t bsel, int o) {
      // lane o / 32 takes the low part of bsel << (o % 32), the next lane what was shifted out
      const int d = lane - (o >> 5);
      mw |= __funnelshift_l(d == 1 ? bsel : 0u, d == 0 ? bsel : 0u, o & 31);
    };
    if (pre) {      // (at most 32 visible rows: one ballot-sized word per head)
      const uint32_t *tg = s_tg + (p - p_lo) * 3;
      place(tg[0], L.m_target);
      if (!no_give) { place(tg[1], L.m_give_target); place(tg[1], L.m_gold_target); }
      if (!tg[2]) mw |= one_bit(L.m_target + L.n_ent);
    } else {
      unsigned any = 0;
      const bool immune = OENT(EA_TIME_ALIVE, p) < c[NC_SPAWN_IMMUNITY];
      #pragma unroll 1
      for (int base = 0; base < n_vis; base += 32) {
        const int i = base + lane;
        bool ok = false, att = false, give = false;
        if (i < n_vis) {
          const int row = vl[i], id = OENT(EA_ID, row), er = OENT(EA_ROW, row), ec = OENT(EA_COL, row);
          const int npc_type = OENT(EA_NPC_TYPE, row);
          ok = nm_linf(er, ec, r0, c0) <= c[NC_REACH] && id != my_id && !(immune && id > 0);
          att = ok && !(no_danger && npc_type > 1);
          // takeru's RewardWrapper.observation zeroes the Give targets anyway (reward_wrapper.py:31-35)
          give = !no_give && n_inv > 0 && er == r0 && ec == c0 && npc_type == 0 && id != my_id;
        }
        any |= __ballot_sync(0xffffffffu, ok);           // the no-op entry is the engine's, before the wrapper edit
        place(__ballot_sync(0xffffffffu, att), L.m_target + base);
        if (!no_give) {
          const unsigned bg = __ballot_sync(0xffffffffu, give);
          place(bg, L.m_give_target + base); place(bg, L.m_gold_target + base);
        }
      }
      if (!any) mw |= one_bit(L.m_target + L.n_ent);
    }
    {
      const bool full = n_inv >= NINV;
      // does a market listing match an ammo stack I own?
      auto ammo_match = [&](int j) -> bool {
        int type = s_mkt[j * IA_N_OBS + IA_TYPE], level = s_mkt[j * IA_N_OBS + IA_LEVEL];
        if (!it_ammo(type) || s_mkt[j * IA_N_OBS + IA_OWNER] == my_id) return false;
        for (int i = 0; i < n_inv; i++) if (OITM(IS_TYPE, inv[i]) == type && OITM(IS_LEVEL, inv[i]) == level) return true;
        return false;
      };
      bool any_ammo = false;
      if (full) { for (int j = lane; j < n_mkt; j += 32) any_ammo |= ammo_match(j); any_ammo = __any_sync(0xffffffffu, any_ammo); }
      if (!(full && !any_ammo))
        #pragma unroll 1
        for (int base = 0; base < n_mkt; base += 32) {
          const int j = base + lane;
          bool ok = false;
          if (j < n_mkt) {
            ok = s_mkt[j * IA_N_OBS + IA_OWNER] != my_id && s_mkt[j * IA_N_OBS + IA_LISTED_PRICE] <= my_gold;
            if (full) ok = ok && ammo_match(j);
          }
          place(__ballot_sync(0xffffffffu, ok), L.m_buy + base);
        }
    }
    if (n_inv > 0) {
      bool b_destroy = false, b_free = false, b_use = false;
      if (lane < n_inv) {
        const int i = inv[lane];
        const bool eq = OITM(IS_EQUIPPED, i) != 0, listed = OITM(IS_PRICE, i) != 0;
        b_destroy = !eq; b_free = !eq && !listed;
        b_use = !listed && OITM(IS_LEVEL, i) <= o_use_level<V>(o, p, OITM(IS_TYPE, i));
      }
      const unsigned bf = __ballot_sync(0xffffffffu, b_free);
      place(__ballot_sync(0xffffffffu, b_destroy), L.m_destroy);
      if (!no_give) place(bf, L.m_give_item);
      place(bf, L.m_sell_item);
      place(__ballot_sync(0xffffffffu, b_use), L.m_use);
    }
    if (!no_give) mw |= range_bits(L.m_gold_price + 1, L.m_gold_price + min(my_gold, L.n_price));
    {
      // North South East West Stay (c_dir_dr / c_dir_dc; computed, a constant-memory look-up by lane would serialise)
      const int ddr = lane == 0 ? -1 : (lane == 1 ? 1 : 0), ddc = lane == 2 ? 1 : (lane == 3 ? -1 : 0);
      const bool mv = lane < 5 && !nm_impassible(tile((r0 + ddr) * S + c0 + ddc));
      place(__ballot_sync(0xffffffffu, mv), L.m_move);
    }
    // RewardWrapper.observation hooks
    // (takeru: Give.InventoryItem[:-1], Give.Target[:-1], GiveGold.Target[:-1], GiveGold.Price[1:]
    //  stay at the template's zeros -- they were never filled in, see no_give above)
    if (wrapper == NW_START_KIT) {
      int prev = 0;
      if (lane == 0) prev = prm.stats[a * ST_N + ST_PREV_PRICE];
      mw &= ~one_bit(L.m_sell_price + __shfl_sync(0xffffffffu, prev, 0));
    }
    // out: 16 mask entries (half a word) become the 16 bytes of one store
    // (at most 1024 entries = 64 stores: two per lane; lane k's come from the words of lanes k / 2 and 16 + k / 2)
#pragma unroll
    for (int half = 0; half < 2; half++) {
      const uint32_t wsrc = __shfl_sync(0xffffffffu, mw, half * 16 + (lane >> 1)) >> ms_shift;
      if (half * 32 + lane < stage_bytes / 16)
        st16(rec + (half * 32 + lane) * 16,
             make_uint4(((wsrc & 15u) * 0x00204081u) & 0x01010101u, (((wsrc >> 4) & 15u) * 0x00204081u) & 0x01010101u,
                        (((wsrc >> 8) & 15u) * 0x00204081u) & 0x01010101u, (((wsrc >> 12) & 15u) * 0x00204081u) & 0x01010101u));
    }
    n_stored += stage_bytes / 16 + 1;
    if (prm.sample_out) {      // queued for the built-in policy (resolved NM_OBS_BATCH agents at a time, top of the loop)
      const uint32_t nz = __ballot_sync(0xffffffffu, mw != 0);
      bb[nb * 33 + lane] = mw;
      if (lane == 0) { bb[nb * 33 + 32] = nz; ba[nb] = (uint16_t)(p - p_lo); }
      nb++;
    }
    // ---- AgentId, CurrentTick ----
    if (lane == 0) st16(rec + L.o_ids, make_uint4(pack2(my_id, tick), 0, 0, 0));
    // ---- Entity rows ----
    // Eight rows (8 x 62 bytes = 31 whole 16-byte chunks) at a time through a per-warp buffer: lane (j, q) copies columns
    // q, q+4, ... of the group's j-th visible row, then 31 lanes store one chunk each.  Rows past n_vis are zeros.
    {
      const int n_chunks = min(nm_align16(L.n_ent * EA_N_OBS * 2) / 16, (max(n_vis, pv) * EA_N_OBS * 2 + 15) / 16);
      n_stored += n_chunks;
      if (V::kStage) {
        // NM_OBS_EROWS rows per group (8: lane = (row, column mod 4), needs the skewed columns to stay free of bank
        // conflicts; 16: lane = (row, column mod 2), half as many groups)
        constexpr int ER = NM_OBS_EROWS, EL = 32 / ER, GC = ER * EA_N_OBS * 2 / 16;      // lanes per row, chunks per group
        const int ej = lane / EL, eq = lane % EL;
        #pragma unroll 1
        for (int g = 0; GC * g < n_chunks; g++) {
          const int i = ER * g + ej;
          int16_t *dst = ebuf + ej * EA_N_OBS + eq;
          if (i < n_vis) {
            const int vr = vl[i];
#pragma unroll
            for (int t = 0; t < (EA_N_OBS + EL - 1) / EL; t++) if (eq + EL * t < EA_N_OBS) dst[EL * t] = OENT(eq + EL * t, vr);
          } else {
#pragma unroll
            for (int t = 0; t < (EA_N_OBS + EL - 1) / EL; t++) if (eq + EL * t < EA_N_OBS) dst[EL * t] = 0;
          }
          __syncwarp();
#pragma unroll
          for (int h = 0; h < (GC + 31) / 32; h++) {
            const int kk = h * 32 + lane, k = GC * g + kk;
            if (kk < GC && k < n_chunks) st16(rec + L.o_entity + k * 16, ((const uint4 *)ebuf)[kk]);
          }
          __syncwarp();
        }
      } else {
        // big family: the table is read in place (HBM / L2), so the chunks are independent of each other and several
        // iterations' loads are in flight: a lane gathers the 8 consecutive int16 of its chunk (at most one row change)
        const int n_el = n_vis * EA_N_OBS;
        #pragma unroll 1
        for (int k = lane; k < n_chunks; k += 32) {
          const int e0 = k * 8;
          uint4 v = zero4;
          if (e0 < n_el) {
            int row = e0 / EA_N_OBS, col = e0 - row * EA_N_OBS;
            int vr = vl[row], vr_next = row + 1 < n_vis ? (int)vl[row + 1] : -1;
            int vals[8];
#pragma unroll
            for (int j = 0; j < 8; j++) {
              vals[j] = vr >= 0 ? (int)OENT(col, vr) : 0;
              if (++col == EA_N_OBS) { col = 0; vr = vr_next; }
            }
            v = make_uint4(pack2(vals[0], vals[1]), pack2(vals[2], vals[3]), pack2(vals[4], vals[5]), pack2(vals[6], vals[7]));
          }
          st16(rec + L.o_entity + k * 16, v);
        }
      }
    }
    // ---- Inventory rows ----
    n_stored += max(n_inv, pi) * 2;
    #pragma unroll 1
    for (int k = lane; k < max(n_inv, pi) * 2; k += 32) {
      int slot = k >> 1;
      uint4 v = zero4;
      if (slot < n_inv) {
        int i = inv[slot];
        int16_t row[IA_N_OBS];
        item_obs_row(c, i, OITM(IS_TYPE, i), OITM(IS_LEVEL, i), OITM(IS_OWNER, i), OITM(IS_QUANTITY, i), OITM(IS_EQUIPPED, i), OITM(IS_PRICE, i), row);
        int h = (k & 1) * 8;
        v = make_uint4(pack2(row[h], row[h + 1]), pack2(row[h + 2], row[h + 3]), pack2(row[h + 4], row[h + 5]), pack2(row[h + 6], row[h + 7]));
      }
      st16(rec + L.o_inventory + k * 16, v);
    }
    // ---- Market block ----
    // one TMA bulk copy from the env's block in shared memory (identical for every agent); rows the record still holds
    // beyond it are zeroed
    n_stored += max(n_mkt, pm) * 2;
    if (lane == 0 && n_mkt > 0) { bulk_s2g(rec + L.o_market, s_mkt, (uint32_t)n_mkt * (IA_N_OBS * 2)); bulk_commit(); }
    #pragma unroll 1
    for (int k = n_mkt * 2 + lane; k < pm * 2; k += 32) st16(rec + L.o_market + k * 16, zero4);
    // ---- Task embedding (constant within an episode) ----
    if (!task_ok) {
      n_stored += L.task_dim * 2 / 16;
      const uint4 *src = (const uint4 *)(prm.embed + (size_t)prm.task_id[a] * L.task_dim);
      for (int k = lane; k < L.task_dim * 2 / 16; k += 32) st16(rec + L.o_task + k * 16, __ldg(src + k));
    }
    // ---- Tile window ----
    // a lane owns 8 consecutive tiles = 24 int16 = three 16-byte stores
    {
      const int n_tiles = tw_tiles, n_groups = tw_groups;
      n_stored += nm_align16(n_tiles * 6) / 16;
      if (tw_fast) {
        if (lane < n_groups) {
          const int w = lane * 8;
          const int rrA = r0 + tw_dr - vis, ccA = c0 + tw_dc - vis;
          // materials of the 8 tiles in order: the rest of window row tw_dr, then the start of the next one
          const uint32_t a8 = fetch8(rrA * S + ccA), b8 = fetch8((rrA + 1) * S + c0 - vis);
          const uint32_t mats = tw_first >= 8 ? a8 : ((a8 & ((1u << (4 * tw_first)) - 1u)) | (b8 << (4 * tw_first)));
          // (row, col) of a tile as one word, col in the high half: tile t of the group is a lane-dependent constant away
          // from the group's first tile; tiles past the end of the window (last group only) are zeros
          const uint32_t rcA = pack2(rrA, ccA), mv = mats & tw_matmask;
          // tiles of the group's second window row: one row down, L.win columns back.  A group holds 8 tiles or (the last
          // one: an odd square is 1 mod 8) a single tile, whose other seven stay zero
          const uint32_t rcA1 = rcA & tw_full, rcN1 = (rcA + 1u - ((uint32_t)L.win << 16)) & tw_full;
          uint32_t rc[8];
          rc[0] = rcA;
#pragma unroll
          for (int t = 1; t < 8; t++) rc[t] = (t >= tw_first ? rcN1 : rcA1) + (uint32_t)t * tw_unit;      // one select, one multiply-add
          // int16 stream row0 col0 mat0 row1 col1 mat1 ... as 12 words; the materials of two tiles are spread into the
          // two halves of one word (y) and merged with the neighbouring row / col halves by byte permutes
          uint32_t wd[12];
#pragma unroll
          for (int u = 0; u < 4; u++) {
            const uint32_t x = (mv >> (8 * u)) & 0xffu;
            const uint32_t y = (x | (x << 12)) & 0x000f000fu;
            wd[3 * u] = rc[2 * u];
            wd[3 * u + 1] = __byte_perm(y, rc[2 * u + 1], 0x5410);
            wd[3 * u + 2] = __byte_perm(rc[2 * u + 1], y, 0x7632);
          }
          uint8_t *dst = rec + L.o_tile + lane * 48;
          const int last = nm_align16(n_tiles * 6);
#pragma unroll
          for (int q = 0; q < 3; q++)
            if (lane * 48 + q * 16 < last) st16(dst + q * 16, make_uint4(wd[4 * q], wd[4 * q + 1], wd[4 * q + 2], wd[4 * q + 3]));
        }
      } else
      #pragma unroll 1
      for (int g = lane; g < n_groups; g += 32) {
        int w = g * 8;
        int dr = w / L.win, dc = w - dr * L.win;
        int v[24];
#pragma unroll
        for (int t = 0; t < 8; t++) {
          bool ok = w + t < n_tiles;
          int rr = r0 + dr - vis, cc = c0 + dc - vis;
          v[3 * t] = ok ? rr : 0; v[3 * t + 1] = ok ? cc : 0; v[3 * t + 2] = ok ? tile(rr * S + cc) : 0;
          if (++dc == L.win) { dc = 0; dr++; }
        }
        uint8_t *dst = rec + L.o_tile + g * 48;
        const int last = nm_align16(n_tiles * 6);      // bytes of the section incl. alignment pad
#pragma unroll
        for (int q = 0; q < 3; q++)
          if (g * 48 + q * 16 < last)
            st16(dst + q * 16, make_uint4(pack2(v[8 * q], v[8 * q + 1]), pack2(v[8 * q + 2], v[8 * q + 3]),
                                          pack2(v[8 * q + 4], v[8 * q + 5]), pack2(v[8 * q + 6], v[8 * q + 7])));
      }
    }
    if (lane == 0) s_meta[p - p_lo] = (uint32_t)n_vis | ((uint32_t)n_inv << 8) | OM_NONZERO | OM_TASK | ((uint32_t)n_mkt << 18);
    __syncwarp();
  }
  if (lane == 0) bulk_wait_all();      // this warp's Market copies have left shared memory and reached the records
  // what the records hold now goes back in one coalesced pass (s_meta entries of agents without work are unchanged)
  __syncthreads();
  #pragma unroll 1
  for (int i = tid; i < p_hi - p_lo; i += T) prm.obs_meta[(size_t)env * P + p_lo + i] = s_meta[i];
  if (!V::kStd && prm.prof && lane == 0) {
    long long t_ = clock64();
    atomicAdd(&prm.prof[40], (unsigned long long)(t_ - w_t0));          // warp-busy cycles in the record loop
    atomicMax(&prm.prof[41 + (blockIdx.x & 7)], (unsigned long long)(t_ - w_t0));
    if (tid == 0) { atomicAdd(&prm.prof[36], (unsigned long long)(t_ - t_prev)); atomicAdd(&prm.prof[37], (unsigned long long)n_work); }
  }
  // bytes this CTA stored (+ the state it pulled in): the kernel's physical traffic estimate
  if (lane == 0) atomicAdd(&prm.counters[4], (unsigned long long)n_stored * 16ULL + ((warp == 0 && p_lo == 0) ? (unsigned long long)(ent_bytes + st_bytes + (uint32_t)(IS_N * 2 * item_hi) + map_bytes) : 0ULL));
}

extern "C" __global__ void __launch_bounds__(NM_OBS_THREADS, NM_OBS_CTAS_PER_SM)
nmmo_obs_kernel(const __grid_constant__ NmParams prm) { obs_body<OSmall>(prm); }

extern "C" __global__ void __launch_bounds__(NM_OBS_THREADS, NM_OBS_CTAS_PER_SM)
nmmo_obs_std_kernel(const __grid_constant__ NmParams prm) { obs_body<OStd>(prm); }

extern "C" __global__ void __launch_bounds__(NM_OBS_THREADS, NM_OBS_CTAS_PER_SM)
nmmo_obs_big_kernel(const __grid_constant__ NmParams prm) { obs_body<OBig>(prm); }

extern "C" __global__ void __launch_bounds__(NM_OBS_THREADS, NM_OBS_CTAS_PER_SM)
nmmo_obs_big_std_kernel(const __grid_constant__ NmParams prm) { obs_body<OBigStd>(prm); }

// ============================================================= action sampler kernel ===
// uniform-random valid action per head from the ActionTargets masks (BASELINE.json config 2:
// "uniform-random valid actions ... counter-based RNG keyed (seed, env, tick, agent, head)").
// One warp per agent: the 946 mask bytes are pulled with 16-byte loads into shared memory,
// then each head is counted and selected with ballots over its mask slice.
extern "C" __global__ void __launch_bounds__(256)
nmmo_sample_kernel(const __grid_constant__ NmParams prm, uint64_t seed, int32_t *out) {
  extern __shared__ __align__(128) uint8_t smem_sampler[];
  const nm_obs_layout &L = prm.L;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
  const int stage_bytes = nm_align16(L.m_end);
  uint8_t *stage = smem_sampler + (size_t)warp * stage_bytes;
  const long long n_agents = (long long)prm.E * prm.P;
  const int off[AC_N] = {L.m_style, L.m_target, L.m_buy, L.m_destroy, L.m_give_item, L.m_give_target,
                         L.m_gold_price, L.m_gold_target, L.m_move, L.m_sell_item, L.m_sell_price, L.m_use};
  const int len[AC_N] = {3, L.n_ent + 1, L.n_mkt + 1, L.n_inv + 1, L.n_inv + 1, L.n_ent + 1, L.n_price,
                         L.n_ent + 1, NM_DIR_N, L.n_inv + 1, L.n_price, L.n_inv + 1};
  const uint32_t *stage32 = (const uint32_t *)stage;
  for (long long a = (long long)blockIdx.x * NW + warp; a < n_agents; a += (long long)gridDim.x * NW) {
    if (!prm.mask[a]) {                       // absent agent: zero record, every head picks 0
      if (lane < AC_N) out[a * AC_N + lane] = 0;
      continue;
    }
    const uint4 *src = (const uint4 *)(prm.obs + (size_t)a * L.stride);
    for (int k = lane; k < stage_bytes / 16; k += 32) ((uint4 *)stage)[k] = __ldcs(src + k);
    __syncwarp();
    const int env = (int)(a / prm.P), p = (int)(a % prm.P);
    const int tick = prm.scalars[(size_t)env * NM_SC_N + SC_TICK];
    // one 64-bit draw per agent, a cheap per-head finaliser on top (nm_action_draw, spec)
    const uint64_t base64 = nm_hash64(seed + (uint64_t)(prm.env_base + env), (uint32_t)tick, RS_ACTION, (uint32_t)p, 0);
    int my_pick = 0;
#pragma unroll
    for (int h = 0; h < AC_N; h++) {
      // mask bytes are 0/1: count them a 32-bit word at a time, clipped to the head's byte range
      const int o0 = off[h];
      int o1 = off[h] + len[h];
      if (h == AC_MOVE_DIR && prm.cfg[NC_SAMPLE_MOVE_PCT] > 0) {      // Move-biased workload, see the observation kernel
        const int nv = (stage[o0] != 0) + (stage[o0 + 1] != 0) + (stage[o0 + 2] != 0) + (stage[o0 + 3] != 0);
        if (nv > 0) {
          if (nm_bounded(nm_action_draw(base64, AC_N), 100) < prm.cfg[NC_SAMPLE_MOVE_PCT]) o1 = o0 + 4;
          else { if (lane == h) my_pick = 4; continue; }
        }
      }
      const int w0 = o0 >> 2, w1 = (o1 + 3) >> 2;
      int total = 0;
      for (int wb = w0; wb < w1; wb += 32) {
        int w = wb + lane;
        uint32_t y = 0;
        if (w < w1) {
          int lo = max(o0 - 4 * w, 0), hi = min(o1 - 4 * w, 4);
          uint32_t bm = (hi >= 4 ? 0xffffffffu : ((1u << (8 * hi)) - 1u)) & ~((1u << (8 * lo)) - 1u);
          y = stage32[w] & 0x01010101u & bm;
        }
        total += __reduce_add_sync(0xffffffffu, __popc(y));
      }
      int pick = 0;
      if (total > 0) {
        int jj = nm_bounded(nm_action_draw(base64, h), total);
        for (int wb = w0; wb < w1; wb += 32) {
          int w = wb + lane;
          uint32_t y = 0;
          if (w < w1) {
            int lo = max(o0 - 4 * w, 0), hi = min(o1 - 4 * w, 4);
            uint32_t bm = (hi >= 4 ? 0xffffffffu : ((1u << (8 * hi)) - 1u)) & ~((1u << (8 * lo)) - 1u);
            y = stage32[w] & 0x01010101u & bm;
          }
          int cnt = __popc(y), incl = cnt;
#pragma unroll
          for (int d = 1; d < 32; d <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += v; }
          int tot = __shfl_sync(0xffffffffu, incl, 31);
          if (jj < tot) {
            bool mine = jj >= incl - cnt && jj < incl;
            int idx = 0;
            if (mine) idx = 4 * w + (int)(__fns(y, 0, jj - (incl - cnt) + 1) >> 3) - o0;
            unsigned who = __ballot_sync(0xffffffffu, mine);
            pick = __shfl_sync(0xffffffffu, idx, __ffs(who) - 1);
            break;
          }
          jj -= tot;
        }
      }
      if (lane == h) my_pick = pick;
    }
    if (lane < AC_N) out[a * AC_N + lane] = my_pick;
    __syncwarp();
  }
}

// ============================================================= forager action source ===
// A scripted survival policy for benchmarking (VERDICT r1 #9): uniform-random agents starve by tick ~35, so long
// runs of the random workload step mostly empty slots.  The forager keeps a population alive for the whole horizon:
// a hungry agent (food or water <= 60) takes the first step of a shortest walkable path, inside its 15x15 tile
// window, to the resource it is shorter of (water: a tile next to water, food: a foliage tile) -- a breadth-first
// search over the window by one warp -- or, seeing none, heads for the map centre; a sated agent stays put; nobody
// fights or trades.  It reads only what a policy reads: the agent's own observation record (tile window, own entity
// row, Move mask).  tests/forager_ref.py is the numpy restatement it is checked against.
extern "C" __global__ void __launch_bounds__(256)
nmmo_forage_kernel(const __grid_constant__ NmParams prm, uint64_t seed, int32_t *out) {
  __shared__ uint8_t s_dist[8][256], s_first[8][256], s_kind[8][256];
  const nm_obs_layout &L = prm.L;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5;
  const long long n_agents = (long long)prm.E * prm.P;
  const int win = L.win, vis = win >> 1, n_tiles = win * win;
  uint8_t *dist = s_dist[warp], *first = s_first[warp], *kind = s_kind[warp];      // kind: bit0 walkable, bit1 goal
  for (long long a = (long long)blockIdx.x * NW + warp; a < n_agents; a += (long long)gridDim.x * NW) {
    const uint8_t *rec = prm.obs + (size_t)a * L.stride;
    const int16_t my_id = *(const int16_t *)(rec + L.o_ids);
    if (!prm.mask[a] || my_id == 0 || n_tiles > 256) {      // absent agent: every head picks 0
      if (lane < AC_N) out[a * AC_N + lane] = 0;
      continue;
    }
    // own row: the Entity row whose id is AgentId
    const int16_t *ent = (const int16_t *)(rec + L.o_entity);
    int food = 0, water = 0, my_r = 0, my_c = 0;
    {
      // (rows are packed at the front of the block and entity ids are never 0: the search stops at the first empty row
      //  instead of touching all 100 -- 6 KB of record per agent, most of this kernel's traffic)
      int found = -1;
      unsigned bm = 0;
      #pragma unroll 1
      for (int base = 0; base < L.n_ent; base += 32) {
        const int r = base + lane;
        const int16_t id = r < L.n_ent ? ent[r * EA_N_OBS + EA_ID] : (int16_t)0;
        bm = __ballot_sync(0xffffffffu, id == my_id);
        if (bm) { found = base + __ffs(bm) - 1; break; }
        if (__ballot_sync(0xffffffffu, id == 0)) break;
      }
      if (bm) { food = ent[found * EA_N_OBS + EA_FOOD]; water = ent[found * EA_N_OBS + EA_WATER];
                my_r = ent[found * EA_N_OBS + EA_ROW]; my_c = ent[found * EA_N_OBS + EA_COL]; }
    }
    const int env = (int)(a / prm.P), p = (int)(a % prm.P);
    const int tick = prm.scalars[(size_t)env * NM_SC_N + SC_TICK];
    const uint64_t base64 = nm_hash64(seed + (uint64_t)(prm.env_base + env), (uint32_t)tick, RS_ACTION, (uint32_t)p, 1);
    const bool hungry = min(food, water) <= 60;
    const int want = water <= food ? MT_WATER : MT_FOILAGE;
    const int16_t *tl = (const int16_t *)(rec + L.o_tile);
    int dir = 4;                       // Stay
    bool decided = !hungry;            // sated: stay where the resources are
    if (hungry) {
      // breadth-first search over the window from the centre tile; the first goal tile reached (ties: lowest window
      // index) gives the first step.  Other entities are ignored (they move).
      const int centre = vis * win + vis;
      __syncwarp();
      for (int w = lane; w < n_tiles; w += 32) {
        const int m = tl[w * 3 + 2];
        const bool walk = !nm_impassible(m);
        bool goal = false;
        if (want == MT_FOILAGE) goal = m == MT_FOILAGE;
        else if (walk) {
          const int r = w / win, c = w % win;
          goal = (r > 0 && tl[(w - win) * 3 + 2] == MT_WATER) || (r < win - 1 && tl[(w + win) * 3 + 2] == MT_WATER) ||
                 (c > 0 && tl[(w - 1) * 3 + 2] == MT_WATER) || (c < win - 1 && tl[(w + 1) * 3 + 2] == MT_WATER);
        }
        kind[w] = (uint8_t)((walk ? 1 : 0) | (goal ? 2 : 0));
        dist[w] = w == centre ? 0 : 255;
        first[w] = 4;
      }
      __syncwarp();
      int hit = (kind[centre] & 2) ? centre : -1;
      for (int round = 1; round <= 48 && hit < 0; round++) {
        bool grew = false;
        int mine = 0x7fffffff;
        for (int w = lane; w < n_tiles; w += 32) {
          if (dist[w] != 255 || !(kind[w] & 1)) continue;
          const int r = w / win, c = w % win;
          // neighbours in the order North, South, West, East of the tile; stepping from a neighbour onto this tile
          int from = -1, step = 4;
          if (r > 0 && dist[w - win] == round - 1) { from = w - win; step = 1; }            // came from the north: moved South
          else if (r < win - 1 && dist[w + win] == round - 1) { from = w + win; step = 0; }
          else if (c > 0 && dist[w - 1] == round - 1) { from = w - 1; step = 2; }            // came from the west: moved East
          else if (c < win - 1 && dist[w + 1] == round - 1) { from = w + 1; step = 3; }
          if (from < 0) continue;
          first[w] = round == 1 ? (uint8_t)step : first[from];
          dist[w] = 254;                 // claimed this round (turned into `round` below, after everybody has looked)
          grew = true;
          if (kind[w] & 2) mine = min(mine, w);
        }
        __syncwarp();
        for (int w = lane; w < n_tiles; w += 32) if (dist[w] == 254) dist[w] = (uint8_t)round;
        __syncwarp();
        mine = __reduce_min_sync(0xffffffffu, mine);
        if (mine != 0x7fffffff) hit = mine;
        if (!__any_sync(0xffffffffu, grew)) break;
      }
      if (hit >= 0) { dir = hit == centre ? 4 : (int)first[hit]; decided = true; }
    }
    if (lane == 0) {
      const int8_t *mv = (const int8_t *)(rec + L.m_move);      // North South East West Stay
      if (!decided) {
        // nothing reachable in sight: head for the map centre (7 ticks in 8), else / when blocked a seeded random valid direction
        const int dr = prm.S / 2 - my_r, dc = prm.S / 2 - my_c;
        if (nm_bounded(nm_action_draw(base64, AC_N), 8) != 0) {
          const int vdir = dr < 0 ? 0 : 1, hdir = dc > 0 ? 2 : 3;
          const int f1 = nm_iabs(dr) >= nm_iabs(dc) ? vdir : hdir, f2 = nm_iabs(dr) >= nm_iabs(dc) ? hdir : vdir;
          if ((f1 < 2 ? dr != 0 : dc != 0) && mv[f1]) { dir = f1; decided = true; }
          else if ((f2 < 2 ? dr != 0 : dc != 0) && mv[f2]) { dir = f2; decided = true; }
        }
        if (!decided) {
          const int nv = (mv[0] != 0) + (mv[1] != 0) + (mv[2] != 0) + (mv[3] != 0);
          if (nv > 0) {
            int j = nm_bounded(nm_action_draw(base64, AC_MOVE_DIR), nv);
            for (int k = 0; k < 4; k++) if (mv[k] && j-- == 0) { dir = k; break; }
          }
        }
      }
      int4 *o4 = (int4 *)(out + a * AC_N);
      // no-op everywhere else: Attack.Target / Give.Target / GiveGold.Target = N_ent, Buy = N_mkt, item heads = N_inv
      o4[0] = make_int4(0, L.n_ent, L.n_mkt, L.n_inv);
      o4[1] = make_int4(L.n_inv, L.n_ent, 0, L.n_ent);
      o4[2] = make_int4(dir, L.n_inv, 0, L.n_inv);
    }
  }
}
