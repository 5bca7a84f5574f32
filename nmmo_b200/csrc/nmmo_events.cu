// nmmo_events.cu -- the event log: the events each env emitted in its last step, as rows in the reference's layout.
//
// With the event log on (nmmo_set_event_log), the step kernel keeps every env's event ring of the call in
// NmParams.ev_log ([E][ev_cap] uint2, in emission order) and its length in ev_n ([E]).  nmmo_events turns the rings of
// an env range into int32 rows [env, ent_id, tick, event, type, level, number, gold, target] (columns 1..8 are the
// columns of the reference's EventLogger), ordered by env, then agent, then emission order, in two launches:
//   nmmo_events_scan_kernel  one CTA: exclusive scan of ev_n over the range -> each env's first row, and the total
//   nmmo_events_kernel       one CTA per env: a stable counting sort of the ring by agent, then one row per thread
// Neither reads anything back to the host.  One agent's events inside a phase come from one thread and phases are
// separated by barriers, so the ring restricted to one agent is in a fixed order; the sort keeps it.
#pragma once

#define NM_EV_THREADS 256
#define NM_EV_SCAN_THREADS 1024

// exclusive prefix sum of one value per thread over the CTA; *total receives the sum (every thread).  s_w: 32 ints
__device__ __forceinline__ int nm_block_excl_scan(int v, int *s_w, int *total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = blockDim.x >> 5;
  int x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += u; }
  if (lane == 31) s_w[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = lane < nw ? s_w[lane] : 0;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) { const int u = __shfl_up_sync(0xffffffffu, w, d); if (lane >= d) w += u; }
    s_w[lane] = w;      // inclusive sums of the warps
  }
  __syncthreads();
  const int r = x - v + (warp ? s_w[warp - 1] : 0);
  *total = s_w[nw - 1];
  __syncthreads();      // s_w is reused by the next call
  return r;
}

// first row of every env of [lo, hi) -> off[env]; rows of the whole range -> count[0]
extern "C" __global__ void __launch_bounds__(NM_EV_SCAN_THREADS) nmmo_events_scan_kernel(const int32_t *ev_n, int lo, int hi,
                                                                                          int32_t *off, int32_t *count) {
  __shared__ int s_w[32];
  int carry = 0;
  for (int b = lo; b < hi; b += NM_EV_SCAN_THREADS) {
    const int e = b + (int)threadIdx.x;
    int total;
    const int x = nm_block_excl_scan(e < hi ? ev_n[e] : 0, s_w, &total);
    if (e < hi) off[e] = carry + x;
    carry += total;
  }
  if (threadIdx.x == 0) count[0] = carry;
}

struct NmEventsArgs {
  const uint2 *ev_log;         // [E][ev_cap]
  const int32_t *ev_n, *off;   // [E]
  const int32_t *scalars;      // [E][NM_SC_N]: SC_TICK
  int ev_cap, P, lo;
  int32_t *rows;               // [cap][9]
  int cap;
};

__constant__ int c_ev_code[17] = {EV_EAT_FOOD, EV_DRINK_WATER, EV_GO_FARTHEST, EV_SCORE_HIT, EV_PLAYER_KILL, EV_CONSUME_ITEM,
                                  EV_GIVE_ITEM, EV_DESTROY_ITEM, EV_HARVEST_ITEM, EV_EQUIP_ITEM, EV_LOOT_ITEM, EV_GIVE_GOLD,
                                  EV_LIST_ITEM, EV_EARN_GOLD, EV_BUY_ITEM, EV_LOOT_GOLD, EV_LEVEL_UP};      // nm_dense_event inverse

// dynamic shared memory: (P + ev_cap) ints
extern "C" __global__ void __launch_bounds__(NM_EV_THREADS) nmmo_events_kernel(const __grid_constant__ NmEventsArgs a) {
  extern __shared__ int s_ev[];
  __shared__ int s_w[32];
  const int env = a.lo + blockIdx.x, tid = threadIdx.x, T = blockDim.x;
  const int n = a.ev_n[env], base = a.off[env];
  if (n == 0 || base >= a.cap) return;      // (uniform over the CTA)
  const uint2 *ev = a.ev_log + (size_t)env * a.ev_cap;
  int *const s_end = s_ev, *const s_idx = s_ev + a.P;
  for (int p = tid; p < a.P; p += T) s_end[p] = 0;
  __syncthreads();
  for (int i = tid; i < n; i += T) atomicAdd(&s_end[ev[i].x & 0xffffu], 1);
  __syncthreads();
  // per-agent counts -> first slot of each agent's bucket
  int carry = 0;
  for (int b = 0; b < a.P; b += T) {
    const int p = b + tid;
    const int c = p < a.P ? s_end[p] : 0;
    int total;
    const int x = nm_block_excl_scan(c, s_w, &total);
    if (p < a.P) s_end[p] = carry + x;
    carry += total;
  }
  __syncthreads();
  // bucket fill in any order (s_end[p] ends as the end of p's bucket = the start of p + 1's), then each bucket sorted
  // by ring index, which restores the emission order
  for (int i = tid; i < n; i += T) s_idx[atomicAdd(&s_end[ev[i].x & 0xffffu], 1)] = i;
  __syncthreads();
  for (int p = tid; p < a.P; p += T) {
    const int s = p ? s_end[p - 1] : 0, e = s_end[p];
    for (int j = s + 1; j < e; j++) {
      const int x = s_idx[j];
      int k = j - 1;
      while (k >= s && s_idx[k] > x) { s_idx[k + 1] = s_idx[k]; k--; }
      s_idx[k + 1] = x;
    }
  }
  __syncthreads();
  const int tick = a.scalars[(size_t)env * NM_SC_N + SC_TICK];
  const int m = min(n, a.cap - base);
  for (int k = tid; k < m; k += T) {
    const uint2 e = ev[s_idx[k]];
    const int de = (e.x >> 16) & 31;
    int number = (int)(int16_t)(e.y & 0xffffu), gold = (int)(int16_t)(e.y >> 16), target = 0;
    // the target's id rides in the half its event leaves zero (emit, nmmo_step.cu)
    if (de == 3 || de == 4 || de == 10) { target = gold; gold = 0; }      // SCORE_HIT, PLAYER_KILL, LOOT_ITEM
    else if (de == 15) { target = number; number = 0; }                 // LOOT_GOLD
    int32_t *r = a.rows + (size_t)(base + k) * 9;
    r[0] = env; r[1] = (int)(e.x & 0xffffu) + 1; r[2] = tick; r[3] = c_ev_code[de]; r[4] = (e.x >> 21) & 31;
    r[5] = (e.x >> 26) & 15; r[6] = number; r[7] = gold; r[8] = target;
  }
}
