// nmmo_rollout.cu -- device-resident rollout storage and GAE (SURVEY.md section 8(f), rank 1).
//
// What it replaces in the reference (reinforcement_learning/clean_pufferl.py):
//   :183-197  the obs / actions / logprobs / rewards / dones / values arrays of batch_size + 1 rows (host)
//   :329-346  per recv(): `indices = where(mask * policy_pool.mask)[: batch_size - ptr + 1]`, seven
//             D2H copies and fancy-index stores, `sort_keys.extend((env_id[i], step))`
//   :413-414  `idxs = sorted(range(len(sort_keys)), key=sort_keys.__getitem__)`
//   :424-436  the batch_size-long Python GAE loop over the sorted samples
//
// Here the batch never leaves the GPU.  A step is appended by a stable stream compaction of the
// alive slots (the records are streamed HBM -> HBM by one warp per row); the (slot, step) sort is a
// counting sort that falls out of the append (a sample's rank inside its slot is the slot's running
// count); the GAE recurrence is evaluated with the reference's float32 operations in the
// reference's order, so advantages are bit-identical to the Python loop: a chain restarts wherever
// `nextnonterminal` is 0 and every chain is walked right-to-left by one warp.
#include <cuda_runtime.h>
#include <stdint.h>
#include <string>
#include <vector>
#include <algorithm>

#include "../../include/nmmo_b200.h"

namespace {

constexpr int RB = 1024;            // threads per block of the scan-shaped kernels

struct RolloutParams {
  int cap;                 // batch_size + 1 rows
  int n_slots;             // agent slots per step (E * P)
  int call_lo, call_n;     // store: the slots [call_lo, call_lo + call_n) of this call (row i of its inputs = slot call_lo + i)
  int stride;              // bytes per observation record (multiple of 16)
  // storage (clean_pufferl.py:183-189)
  uint8_t *obs; int32_t *actions; float *logprobs, *rewards, *dones, *values;
  int32_t *slot, *rank, *step;     // sort key (slot, step) and the sample's rank inside its slot
  int32_t *count;          // [n_slots] samples stored per slot
  int32_t *base;           // [n_slots] exclusive prefix of count
  int32_t *blocksum;       // scratch for the two-level scans
  int32_t *d_ptr;          // [4]: ptr, total selected this step, n_starts, spare
  int32_t *idxs;           // [cap] sample indices in (slot, step) order
  float *delta, *coef, *adv;       // [cap]
  int32_t *starts;         // [cap] chain start positions
  // compact mode (nmmo_rollout_create_compact): a row keeps the record without its Market and Task sections.  The Market
  // block is identical for every agent of an env in a step and is stored once per (step, env); the Task block is the
  // embedding of the agent's task and is stored as the task id.  nmmo_rollout_expand re-assembles full records.
  int compact;             // 0 = rows are whole records
  int agents_per_env, n_envs;
  int m_off, m_len, t_off, t_len;  // byte ranges of the two sections inside a record (multiples of 16)
  int ids_off;             // byte offset of the int16 AgentId: 0 there = the all-zero record of an agent that just died
  int row_stride;          // bytes per stored row (= stride - m_len - t_len in compact mode)
  int max_steps;           // Market blocks: max_steps * n_envs of m_len bytes
  uint8_t *market;
  int32_t *mslot;          // [cap] row -> Market block (blocks stored by earlier calls + env of the call)
  int32_t *task;           // [cap] row -> task id
};

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) { int u = __shfl_up_sync(0xffffffffu, v, d); if (lane >= d) v += u; }
  return v;
}
// exclusive scan of one value per thread across a 1024-thread block; returns the block total in `total`
__device__ int block_excl_scan(int v, int *s_warp, int &total) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int incl = warp_incl_scan(v, lane);
  if (lane == 31) s_warp[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = s_warp[lane];
    int wi = warp_incl_scan(w, lane);
    s_warp[lane] = wi - w;
    if (lane == 31) s_warp[32] = wi;
  }
  __syncthreads();
  total = s_warp[32];
  int r = s_warp[warp] + incl - v;
  __syncthreads();
  return r;
}

__device__ __forceinline__ bool selected(const RolloutParams &p, const uint8_t *mask, const uint8_t *learner, int i) {
  return i < p.call_n && mask[i] != 0 && (learner == nullptr || learner[i] != 0);
}

// ---- append: pass 1, selected slots per 1024-slot block --------------------------------------
__global__ void __launch_bounds__(RB) k_store_count(RolloutParams p, const uint8_t *mask, const uint8_t *learner) {
  __shared__ int s_warp[33];
  int i = blockIdx.x * RB + threadIdx.x, total;
  block_excl_scan(selected(p, mask, learner, i) ? 1 : 0, s_warp, total);
  if (threadIdx.x == 0) p.blocksum[blockIdx.x] = total;
}
// ---- exclusive scan of the block sums by one block (n <= 1024 * 1024 entries), in place --------
__global__ void __launch_bounds__(RB) k_scan_blocks(int32_t *v, int n, int32_t *total_out) {
  __shared__ int s_warp[33];
  int carry = 0;
  for (int b0 = 0; b0 < n; b0 += RB) {
    int i = b0 + threadIdx.x, x = i < n ? v[i] : 0, total;
    int ex = block_excl_scan(x, s_warp, total);
    if (i < n) v[i] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0 && total_out) *total_out = carry;
}
// ---- append: pass 2, scalars + keys, then the records (one warp per selected row) --------------
__global__ void __launch_bounds__(RB) k_store_rows(RolloutParams p, const uint8_t *obs, const int32_t *actions,
                                                  const float *logprob, const float *value, const float *reward,
                                                  const float *done, const uint8_t *mask, const uint8_t *learner, int step) {
  __shared__ int s_warp[33];
  __shared__ int s_src[RB], s_dst[RB];
  __shared__ int s_n;
  const int i = blockIdx.x * RB + threadIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool sel = selected(p, mask, learner, i);
  int total;
  const int rank = block_excl_scan(sel ? 1 : 0, s_warp, total);
  const int pos = p.d_ptr[0] + p.blocksum[blockIdx.x] + rank;       // clean_pufferl.py:337-339
  const bool keep = sel && pos < p.cap;                              // `[: batch_size - ptr + 1]`
  if (threadIdx.x == 0) s_n = 0;
  __syncthreads();
  if (keep) {
    const int4 *a4 = (const int4 *)(actions + (size_t)i * 12);
    int4 *o4 = (int4 *)(p.actions + (size_t)pos * 12);
    o4[0] = a4[0]; o4[1] = a4[1]; o4[2] = a4[2];
    p.logprobs[pos] = logprob[i]; p.values[pos] = value[i]; p.rewards[pos] = reward[i]; p.dones[pos] = done[i];
    const int g = p.call_lo + i;
    p.slot[pos] = g; p.step[pos] = step;
    p.rank[pos] = p.count[g];                 // steps arrive in order: the running count is the rank
    p.count[g] += 1;
    int k = atomicAdd(&s_n, 1);
    s_src[k] = i; s_dst[k] = pos;
  }
  __syncthreads();
  const int n = s_n, n16 = p.stride >> 4;
  if (!p.compact) {
    for (int k = warp; k < n; k += RB / 32) {
      const uint4 *src = (const uint4 *)(obs + (size_t)s_src[k] * p.stride);
      uint4 *dst = (uint4 *)(p.obs + (size_t)s_dst[k] * p.stride);
      for (int q = lane; q < n16; q += 32) __stcs(dst + q, __ldcs(src + q));
    }
  } else {
    // the record minus its Market and Task sections, packed
    const int m0 = p.m_off >> 4, m1 = (p.m_off + p.m_len) >> 4, t0 = p.t_off >> 4, t1 = (p.t_off + p.t_len) >> 4;
    for (int k = warp; k < n; k += RB / 32) {
      const uint4 *src = (const uint4 *)(obs + (size_t)s_src[k] * p.stride);
      uint4 *dst = (uint4 *)(p.obs + (size_t)s_dst[k] * p.row_stride);
      for (int q = lane; q < n16; q += 32) {
        if ((q >= m0 && q < m1) || (q >= t0 && q < t1)) continue;
        const int skipped = (q >= m1 ? m1 - m0 : 0) + (q >= t1 ? t1 - t0 : 0);      // (sections in either order)
        __stcs(dst + q - skipped, __ldcs(src + q));
      }
    }
  }
}
// compact mode: per kept row the Market block and the task id; per env of the call the Market block of its first selected
// agent, at block mbase + env
__device__ __forceinline__ bool zero_record(const RolloutParams &p, const uint8_t *obs, int i) {
  return *(const int16_t *)(obs + (size_t)i * p.stride + p.ids_off) == 0;
}
__global__ void __launch_bounds__(RB) k_store_compact_keys(RolloutParams p, const uint8_t *obs, const uint8_t *mask, const uint8_t *learner,
                                                          const int32_t *task_id, int mbase) {
  __shared__ int s_warp[33];
  const int i = blockIdx.x * RB + threadIdx.x;
  const bool sel = selected(p, mask, learner, i);
  int total;
  const int rank = block_excl_scan(sel ? 1 : 0, s_warp, total);
  const int pos = p.d_ptr[0] + p.blocksum[blockIdx.x] + rank;
  if (sel && pos < p.cap) {
    // an agent that died this tick is stored with the all-zero record: its Market and Task sections are zeros too (-1)
    const bool z = zero_record(p, obs, i);
    p.mslot[pos] = z ? -1 : mbase + i / p.agents_per_env;
    p.task[pos] = z ? -1 : task_id[i];
  }
}
__global__ void __launch_bounds__(256) k_store_market(RolloutParams p, const uint8_t *obs, const uint8_t *mask, const uint8_t *learner,
                                                     int mbase) {
  const int lane = threadIdx.x & 31, env = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (env >= p.call_n / p.agents_per_env) return;
  int first = -1;
  for (int b = 0; b < p.agents_per_env && first < 0; b += 32) {
    const int a = b + lane;
    const unsigned m = __ballot_sync(0xffffffffu, a < p.agents_per_env && selected(p, mask, learner, env * p.agents_per_env + a) &&
                                                       !zero_record(p, obs, env * p.agents_per_env + a));
    if (m) first = b + __ffs(m) - 1;
  }
  if (first < 0) return;                      // nobody of this env is stored this step
  const uint4 *src = (const uint4 *)(obs + (size_t)(env * p.agents_per_env + first) * p.stride + p.m_off);
  uint4 *dst = (uint4 *)(p.market + ((size_t)mbase + env) * p.m_len);
  for (int q = lane; q < (p.m_len >> 4); q += 32) __stcs(dst + q, __ldcs(src + q));
}
// re-assemble full records: out[k] = row idxs[k] (or row k when idxs is NULL) with its Market block and Task embedding
__global__ void __launch_bounds__(256) k_expand(RolloutParams p, const int32_t *idxs, int n, const uint16_t *embed, uint8_t *out) {
  const int lane = threadIdx.x & 31;
  const int m0 = p.m_off >> 4, m1 = (p.m_off + p.m_len) >> 4, t0 = p.t_off >> 4, t1 = (p.t_off + p.t_len) >> 4, n16 = p.stride >> 4;
  for (int k = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; k < n; k += (gridDim.x * blockDim.x) >> 5) {
    const int row = idxs ? idxs[k] : k;
    const uint4 *src = (const uint4 *)(p.obs + (size_t)row * p.row_stride);
    const bool z = p.mslot[row] < 0;
    const uint4 *mk = (const uint4 *)(p.market + (size_t)max(p.mslot[row], 0) * p.m_len);
    const uint4 *tk = (const uint4 *)(embed + (size_t)max(p.task[row], 0) * (p.t_len >> 1));
    uint4 *dst = (uint4 *)(out + (size_t)k * p.stride);
    for (int q = lane; q < n16; q += 32) {
      uint4 v;
      if (q >= m0 && q < m1) v = z ? make_uint4(0, 0, 0, 0) : __ldg(mk + q - m0);
      else if (q >= t0 && q < t1) v = z ? make_uint4(0, 0, 0, 0) : __ldg(tk + q - t0);
      else v = __ldcs(src + q - ((q >= m1 ? m1 - m0 : 0) + (q >= t1 ? t1 - t0 : 0)));
      __stcs(dst + q, v);
    }
  }
}
__global__ void k_advance_ptr(RolloutParams p) {
  if (threadIdx.x == 0) p.d_ptr[0] = min(p.cap, p.d_ptr[0] + p.d_ptr[1]);
}

// ---- counting sort by (slot, step) ------------------------------------------------------------
__global__ void __launch_bounds__(RB) k_count_sums(RolloutParams p) {
  __shared__ int s_warp[33];
  int i = blockIdx.x * RB + threadIdx.x, total;
  block_excl_scan(i < p.n_slots ? p.count[i] : 0, s_warp, total);
  if (threadIdx.x == 0) p.blocksum[blockIdx.x] = total;
}
__global__ void __launch_bounds__(RB) k_count_base(RolloutParams p) {
  __shared__ int s_warp[33];
  int i = blockIdx.x * RB + threadIdx.x, total;
  int ex = block_excl_scan(i < p.n_slots ? p.count[i] : 0, s_warp, total);
  if (i < p.n_slots) p.base[i] = p.blocksum[blockIdx.x] + ex;
}
__global__ void k_scatter_idxs(RolloutParams p) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < p.d_ptr[0]) p.idxs[p.base[p.slot[j]] + p.rank[j]] = j;
}

// ---- GAE (clean_pufferl.py:424-436) -------------------------------------------------------------
// delta[t] and the chain coefficient, with the reference's float32 operations in its order:
//   nextnonterminal = 1.0 - dones[i_nxt]
//   delta = rewards[i_nxt] + gamma * values[i_nxt] * nextnonterminal - values[i]
//   advantages[t] = lastgaelam = delta + gamma * gae_lambda * nextnonterminal * lastgaelam
__global__ void k_gae_prepare(RolloutParams p, float gamma_f, float gl_f) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = p.d_ptr[0] - 1;
  if (t == 0 && blockIdx.x == 0) p.d_ptr[2] = 0;
  if (t >= n) return;
  const int i = p.idxs[t], j = p.idxs[t + 1];
  const float nnt = __fsub_rn(1.0f, p.dones[j]);
  const float d = __fsub_rn(__fadd_rn(p.rewards[j], __fmul_rn(__fmul_rn(gamma_f, p.values[j]), nnt)), p.values[i]);
  p.delta[t] = d;
  p.coef[t] = __fmul_rn(gl_f, nnt);
}
// a chain starts at the last sample and wherever the coefficient is exactly 0 (nextnonterminal == 0)
__global__ void k_gae_starts(RolloutParams p) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int n = p.d_ptr[0] - 1;
  if (t >= n) return;
  if (t == n - 1 || p.coef[t] == 0.0f) p.starts[atomicAdd(&p.d_ptr[2], 1)] = t;
}
// one warp per chain, right to left; lanes fetch 32 elements at a time, the recurrence itself is
// the reference's two float32 operations per element (multiply, then add; never fused)
__global__ void k_gae_chains(RolloutParams p) {
  const int lane = threadIdx.x & 31;
  const int wid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, nw = (gridDim.x * blockDim.x) >> 5;
  const int n_starts = p.d_ptr[2];
  for (int s = wid; s < n_starts; s += nw) {
    const int t0 = p.starts[s];
    float last = 0.0f;
    bool open = true;
    for (int hi = t0; hi >= 0 && open; hi -= 32) {
      const int t = hi - lane;
      float d = 0.0f, c = 0.0f;
      if (t >= 0) { d = p.delta[t]; c = p.coef[t]; }
      // the chain ends before the next start to the left (coefficient 0), which is another warp's
      const bool stop = t < 0 || (t != t0 && c == 0.0f);
      const unsigned stopm = __ballot_sync(0xffffffffu, stop);
      const int len = stopm ? __ffs(stopm) - 1 : 32;
      float mine = 0.0f;
      for (int k = 0; k < len; k++) {
        const float dk = __shfl_sync(0xffffffffu, d, k), ck = __shfl_sync(0xffffffffu, c, k);
        last = (hi - k == t0) ? dk : __fadd_rn(dk, __fmul_rn(ck, last));
        if (lane == k) mine = last;
      }
      if (lane < len) p.adv[t] = mine;
      open = len == 32;
    }
  }
}

}  // namespace

// ======================================================================== C ABI ================
struct nmmo_rollout {
  RolloutParams p;
  int device;
  int n_mblocks = 0;       // compact mode: Market blocks stored since the last reset
  std::vector<void *> allocs;
};

static thread_local std::string g_rerr;
extern "C" const char *nmmo_rollout_last_error(void) { return g_rerr.c_str(); }
static int rfail(int code, const std::string &m) { g_rerr = m; return code; }
#define RCU(call)                                                                                  \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess) return rfail(NM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

template <typename T>
static int ralloc(nmmo_rollout *r, T **ptr, size_t count) {
  void *q = nullptr;
  size_t bytes = std::max<size_t>(count * sizeof(T), 16);
  RCU(cudaMalloc(&q, bytes));
  RCU(cudaMemset(q, 0, bytes));
  r->allocs.push_back(q);
  *ptr = (T *)q;
  return 0;
}
#define RA(ptr, count) do { int rc_ = ralloc(r, &(ptr), (count)); if (rc_) { nmmo_rollout_destroy(r); return rc_; } } while (0)

extern "C" int nmmo_rollout_destroy(nmmo_rollout *r) {
  if (!r) return NM_OK;
  cudaSetDevice(r->device);
  cudaDeviceSynchronize();
  for (void *q : r->allocs) cudaFree(q);
  delete r;
  return NM_OK;
}

static int rollout_create(int device, int batch_size, int n_slots, int obs_stride, int agents_per_env, int m_off, int m_len,
                          int t_off, int t_len, int ids_off, int max_steps, nmmo_rollout **out);

extern "C" int nmmo_rollout_create(int device, int batch_size, int n_slots, int obs_stride, nmmo_rollout **out) {
  return rollout_create(device, batch_size, n_slots, obs_stride, 0, 0, 0, 0, 0, 0, 0, out);
}

extern "C" int nmmo_rollout_create_compact(int device, int batch_size, int n_slots, int obs_stride, int agents_per_env,
                                           int market_off, int market_bytes, int task_off, int task_bytes, int ids_off, int max_steps,
                                           nmmo_rollout **out) {
  if (agents_per_env <= 0 || n_slots % std::max(agents_per_env, 1) || max_steps <= 0 || market_bytes <= 0 || task_bytes <= 0 ||
      ((market_off | market_bytes | task_off | task_bytes) & 15) || market_off + market_bytes > obs_stride || task_off + task_bytes > obs_stride ||
      !(market_off + market_bytes <= task_off || task_off + task_bytes <= market_off))
    return rfail(NM_ERR_ARG, "compact rollout: sections must be 16-byte aligned, disjoint and inside the record; n_slots a multiple of agents_per_env");
  if (ids_off < 0 || ids_off + 2 > obs_stride) return rfail(NM_ERR_ARG, "compact rollout: bad AgentId offset");
  return rollout_create(device, batch_size, n_slots, obs_stride, agents_per_env, market_off, market_bytes, task_off, task_bytes, ids_off, max_steps, out);
}

static int rollout_create(int device, int batch_size, int n_slots, int obs_stride, int agents_per_env, int m_off, int m_len,
                          int t_off, int t_len, int ids_off, int max_steps, nmmo_rollout **out) {
  if (!out || batch_size <= 0 || n_slots <= 0 || obs_stride <= 0 || (obs_stride & 15))
    return rfail(NM_ERR_ARG, "batch_size, n_slots must be positive and obs_stride a positive multiple of 16");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return rfail(NM_ERR_CUDA, "no CUDA device: no CPU fallback");
  if (device < 0 || device >= ndev) return rfail(NM_ERR_ARG, "bad device index");
  RCU(cudaSetDevice(device));
  nmmo_rollout *r = new nmmo_rollout();
  r->device = device;
  RolloutParams &p = r->p;
  p.cap = batch_size + 1; p.n_slots = n_slots; p.stride = obs_stride;
  p.compact = agents_per_env > 0; p.agents_per_env = agents_per_env; p.n_envs = p.compact ? n_slots / agents_per_env : 0;
  p.m_off = m_off; p.m_len = m_len; p.t_off = t_off; p.t_len = t_len; p.ids_off = ids_off; p.max_steps = max_steps;
  p.row_stride = obs_stride - m_len - t_len;
  size_t cap = (size_t)p.cap;
  if (p.compact) { RA(p.market, (size_t)max_steps * p.n_envs * m_len); RA(p.mslot, cap); RA(p.task, cap); }
  RA(p.obs, cap * p.row_stride); RA(p.actions, cap * 12); RA(p.logprobs, cap); RA(p.rewards, cap); RA(p.dones, cap); RA(p.values, cap);
  RA(p.slot, cap); RA(p.rank, cap); RA(p.step, cap); RA(p.count, (size_t)n_slots); RA(p.base, (size_t)n_slots);
  RA(p.blocksum, (size_t)(n_slots + RB - 1) / RB + 1); RA(p.d_ptr, 4); RA(p.idxs, cap);
  RA(p.delta, cap); RA(p.coef, cap); RA(p.adv, cap); RA(p.starts, cap);
  *out = r;
  return NM_OK;
}

extern "C" int nmmo_rollout_reset(nmmo_rollout *r, void *stream) {
  if (!r) return rfail(NM_ERR_ARG, "null handle");
  RCU(cudaSetDevice(r->device));
  cudaStream_t st = (cudaStream_t)stream;
  RCU(cudaMemsetAsync(r->p.count, 0, sizeof(int32_t) * r->p.n_slots, st));
  RCU(cudaMemsetAsync(r->p.d_ptr, 0, sizeof(int32_t) * 4, st));
  r->n_mblocks = 0;
  return NM_OK;
}

extern "C" int nmmo_rollout_store_range(nmmo_rollout *r, int slot_lo, int n, const uint8_t *obs, const int32_t *actions,
                                        const float *logprob, const float *value, const float *reward, const float *done,
                                        const uint8_t *mask, const uint8_t *learner_mask, const int32_t *task_id, int step,
                                        void *stream) {
  if (!r || !obs || !actions || !logprob || !value || !reward || !done || !mask) return rfail(NM_ERR_ARG, "null argument");
  if (((uintptr_t)obs | (uintptr_t)actions) & 15) return rfail(NM_ERR_ARG, "obs and actions must be 16-byte aligned");
  if (slot_lo < 0 || n <= 0 || n > r->p.n_slots - slot_lo) return rfail(NM_ERR_ARG, "slot range must satisfy 0 <= slot_lo < slot_lo + n <= n_slots");
  RolloutParams p = r->p;
  p.call_lo = slot_lo; p.call_n = n;
  int mbase = 0;
  if (p.compact) {
    if (!task_id) return rfail(NM_ERR_ARG, "compact store needs the task ids");
    if (slot_lo % p.agents_per_env || n % p.agents_per_env) return rfail(NM_ERR_ARG, "compact store: the slot range must cover whole envs");
    if (r->n_mblocks + n / p.agents_per_env > p.max_steps * p.n_envs)
      return rfail(NM_ERR_LIMIT, "compact rollout: the Market store is full (more than max_steps whole-handle store calls since the last reset)");
    mbase = r->n_mblocks;
  } else if (task_id) return rfail(NM_ERR_ARG, "task ids are for compact rollouts only");
  RCU(cudaSetDevice(r->device));
  cudaStream_t st = (cudaStream_t)stream;
  int nb = (n + RB - 1) / RB;
  k_store_count<<<nb, RB, 0, st>>>(p, mask, learner_mask);
  k_scan_blocks<<<1, RB, 0, st>>>(p.blocksum, nb, p.d_ptr + 1);
  if (p.compact) {
    k_store_compact_keys<<<nb, RB, 0, st>>>(p, obs, mask, learner_mask, task_id, mbase);
    k_store_market<<<(n / p.agents_per_env * 32 + 255) / 256, 256, 0, st>>>(p, obs, mask, learner_mask, mbase);
    r->n_mblocks += n / p.agents_per_env;
  }
  k_store_rows<<<nb, RB, 0, st>>>(p, obs, actions, logprob, value, reward, done, mask, learner_mask, step);
  k_advance_ptr<<<1, 32, 0, st>>>(p);
  RCU(cudaGetLastError());
  return NM_OK;
}

extern "C" int nmmo_rollout_store(nmmo_rollout *r, const uint8_t *obs, const int32_t *actions, const float *logprob,
                                  const float *value, const float *reward, const float *done, const uint8_t *mask,
                                  const uint8_t *learner_mask, int step, void *stream) {
  if (r && r->p.compact) return rfail(NM_ERR_STATE, "compact rollout: use nmmo_rollout_store_compact (needs the task ids)");
  if (!r) return rfail(NM_ERR_ARG, "null argument");
  return nmmo_rollout_store_range(r, 0, r->p.n_slots, obs, actions, logprob, value, reward, done, mask, learner_mask, nullptr, step, stream);
}

extern "C" int nmmo_rollout_store_compact(nmmo_rollout *r, const uint8_t *obs, const int32_t *actions, const float *logprob,
                                          const float *value, const float *reward, const float *done, const uint8_t *mask,
                                          const uint8_t *learner_mask, const int32_t *task_id, int step, void *stream) {
  if (!r || !r->p.compact || !task_id) return rfail(NM_ERR_ARG, "compact store needs a compact rollout and the task ids");
  return nmmo_rollout_store_range(r, 0, r->p.n_slots, obs, actions, logprob, value, reward, done, mask, learner_mask, task_id, step, stream);
}

extern "C" int nmmo_rollout_ptr(nmmo_rollout *r, void *stream, int *ptr_out) {
  if (!r || !ptr_out) return rfail(NM_ERR_ARG, "null argument");
  RCU(cudaSetDevice(r->device));
  int32_t v = 0;
  RCU(cudaMemcpyAsync(&v, r->p.d_ptr, sizeof(v), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  RCU(cudaStreamSynchronize((cudaStream_t)stream));
  *ptr_out = v;
  return NM_OK;
}

extern "C" int nmmo_rollout_gae(nmmo_rollout *r, double gamma, double gae_lambda, void *stream) {
  if (!r) return rfail(NM_ERR_ARG, "null handle");
  RCU(cudaSetDevice(r->device));
  cudaStream_t st = (cudaStream_t)stream;
  const RolloutParams &p = r->p;
  int nb = (p.n_slots + RB - 1) / RB;
  k_count_sums<<<nb, RB, 0, st>>>(p);
  k_scan_blocks<<<1, RB, 0, st>>>(p.blocksum, nb, nullptr);
  k_count_base<<<nb, RB, 0, st>>>(p);
  int cb = (p.cap + 255) / 256;
  k_scatter_idxs<<<cb, 256, 0, st>>>(p);
  // a Python float times a float32 tensor is a float32 multiply by the rounded scalar
  k_gae_prepare<<<cb, 256, 0, st>>>(p, (float)gamma, (float)(gamma * gae_lambda));
  k_gae_starts<<<cb, 256, 0, st>>>(p);
  k_gae_chains<<<148 * 4, 256, 0, st>>>(p);
  RCU(cudaGetLastError());
  return NM_OK;
}

extern "C" int nmmo_rollout_expand(nmmo_rollout *r, const int32_t *idxs_dev, int n, const uint16_t *task_embed_dev, uint8_t *out_dev, void *stream) {
  if (!r || !r->p.compact || !task_embed_dev || !out_dev || n < 0) return rfail(NM_ERR_ARG, "expand needs a compact rollout, the embedding table and an output buffer");
  if ((uintptr_t)out_dev & 15) return rfail(NM_ERR_ARG, "output must be 16-byte aligned");
  RCU(cudaSetDevice(r->device));
  if (n == 0) return NM_OK;
  k_expand<<<std::min((n * 32 + 255) / 256, 148 * 16), 256, 0, (cudaStream_t)stream>>>(r->p, idxs_dev, n, task_embed_dev, out_dev);
  RCU(cudaGetLastError());
  return NM_OK;
}

extern "C" void *nmmo_rollout_buffer(nmmo_rollout *r, int which) {
  if (!r) return nullptr;
  const RolloutParams &p = r->p;
  switch (which) {
    case NM_RB_OBS: return p.obs; case NM_RB_ACTIONS: return p.actions; case NM_RB_LOGPROBS: return p.logprobs;
    case NM_RB_REWARDS: return p.rewards; case NM_RB_DONES: return p.dones; case NM_RB_VALUES: return p.values;
    case NM_RB_SLOT: return p.slot; case NM_RB_STEP: return p.step; case NM_RB_IDXS: return p.idxs;
    case NM_RB_ADVANTAGES: return p.adv;
    case NM_RB_MARKET: return p.market; case NM_RB_MARKET_SLOT: return p.mslot; case NM_RB_TASK_ID: return p.task;
  }
  return nullptr;
}
