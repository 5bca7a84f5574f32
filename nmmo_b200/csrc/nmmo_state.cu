// nmmo_state.cu -- save environments to device blobs and load them into any slot of a compatible handle.
//
// One blob per env, state_bytes long (a multiple of 128): a 128-byte header, then one 16-byte-aligned section per
// per-env buffer that a step reads and an earlier step or reset wrote (DESIGN.md 2.3; the host side builds the
// section table in nmmo_create, nmmo_api.cu state_layout).  Every CTA copies one chunk of one env's blob, so a save
// or load of many envs spreads over the whole GPU whatever the section sizes are.  Sections whose tail is dead in the
// handle (the item columns above SC_ITEM_HI, the depleted-tile list beyond SC_N_DEPL, the danger stack above
// SC_N_DANGER) move only their live prefix; save writes zeros over the rest, so that blobs of equal states are
// byte-equal (up to the order of the depleted-tile list, which the step kernel fills with atomics and keeps unordered)
// and a save right after a load returns the loaded bytes.
#pragma once

#define NM_STATE_MAGIC 0x54534d4eu      // "NMST"
#define NM_STATE_VERSION 1u
#define NM_STATE_HEADER 128
#define NM_STATE_MAX_SECS 32
#define NM_STATE_IDS 512                // env ids per launch (they travel as kernel parameters)
#define NM_STATE_CHUNK 32768            // blob bytes per CTA
#define NM_STATE_THREADS 256

struct NmStateHeader {                  // the first bytes of every blob; the rest of the 128 are zero
  uint32_t magic, version, family, reserved;
  uint64_t state_bytes, digest;
};

struct NmStateSec {
  uint8_t *h;             // handle buffer of env 0
  uint32_t h_env;         // bytes between two envs in the handle buffer
  uint32_t b_off, bytes;  // where the section sits in the blob, and its size
  uint32_t span;          // bytes up to the next section (its padding is zeroed by save)
  int16_t live_sc, unit;  // live prefix = clamp(scalars[live_sc], 0, bytes / unit) * unit bytes; live_sc < 0: all of it
};

struct NmStateArgs {
  NmStateSec sec[NM_STATE_MAX_SECS];
  int n_sec;
  uint32_t state_bytes, n_chunks, sc_off;      // sc_off: blob offset of the scalars section
  const int32_t *scalars;                      // save: the handle's scalars (live prefixes)
  uint32_t *obs_meta;                          // load: OM_TASK is cleared for the loaded envs' agents
  int32_t *ev_n;                               // load, event log on: the loaded envs have no events
  int P;
  NmStateHeader hdr;
  int n;
  int32_t ids[NM_STATE_IDS];
};

// [0, n) bytes; dst and src 16-byte aligned (or not: then 4-byte or byte copies)
__device__ __forceinline__ void nm_state_copy(uint8_t *dst, const uint8_t *src, uint32_t n) {
  const int t = threadIdx.x, T = blockDim.x;
  const uintptr_t al = (uintptr_t)dst | (uintptr_t)src;
  uint32_t done = 0;
  if ((al & 15) == 0) {
    const uint32_t n16 = n >> 4;
    const uint4 *s4 = (const uint4 *)src;
    uint4 *d4 = (uint4 *)dst;
    #pragma unroll 4
    for (uint32_t i = t; i < n16; i += T) d4[i] = s4[i];
    done = n16 << 4;
  } else if ((al & 3) == 0) {
    const uint32_t n4 = n >> 2;
    for (uint32_t i = t; i < n4; i += T) ((uint32_t *)dst)[i] = ((const uint32_t *)src)[i];
    done = n4 << 2;
  }
  for (uint32_t i = done + t; i < n; i += T) dst[i] = src[i];
}

// zeros over [0, n) bytes of a blob (the start may sit anywhere in a 16-byte word)
__device__ __forceinline__ void nm_state_zero(uint8_t *dst, uint32_t n) {
  const int t = threadIdx.x, T = blockDim.x;
  const uint32_t head = min(n, (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15));
  for (uint32_t i = t; i < head; i += T) dst[i] = 0;
  const uint32_t n16 = (n - head) >> 4;
  uint4 *d4 = (uint4 *)(dst + head);
  #pragma unroll 4
  for (uint32_t i = t; i < n16; i += T) d4[i] = make_uint4(0, 0, 0, 0);
  for (uint32_t i = head + (n16 << 4) + t; i < n; i += T) dst[i] = 0;
}

template <bool SAVE>
__device__ __forceinline__ void state_body(const NmStateArgs &a, uint8_t *blobs) {
  const int j = blockIdx.x / a.n_chunks, c = blockIdx.x % a.n_chunks;
  if (j >= a.n) return;
  const int env = a.ids[j];
  uint8_t *blob = blobs + (size_t)j * a.state_bytes;
  const int32_t *sc = SAVE ? a.scalars + (size_t)env * NM_SC_N : (const int32_t *)(blob + a.sc_off);
  const uint32_t c0 = (uint32_t)c * NM_STATE_CHUNK, c1 = min(c0 + NM_STATE_CHUNK, a.state_bytes);
  if (c == 0) {
    if (SAVE) {
      const int t = threadIdx.x;
      if (t < NM_STATE_HEADER / 4) {
        uint32_t w = 0;
        if (t < (int)(sizeof(NmStateHeader) / 4)) w = ((const uint32_t *)&a.hdr)[t];
        ((uint32_t *)blob)[t] = w;
      }
    } else {
      // the Task block of the slot's records may hold another task: the observation pass after the load rewrites it
      for (int i = threadIdx.x; i < a.P; i += blockDim.x) a.obs_meta[(size_t)env * a.P + i] &= ~OM_TASK;
      if (a.ev_n && threadIdx.x == 0) a.ev_n[env] = 0;
    }
  }
  for (int s = 0; s < a.n_sec; s++) {
    const NmStateSec &q = a.sec[s];
    const uint32_t x0 = max(c0, q.b_off), x1 = min(c1, q.b_off + q.span);
    if (x0 >= x1) continue;
    uint32_t live = q.bytes;
    if (q.live_sc >= 0) live = (uint32_t)min(max(sc[q.live_sc], 0), (int)(q.bytes / q.unit)) * q.unit;
    const uint32_t r0 = x0 - q.b_off, r1 = x1 - q.b_off, rl = min(r1, live);
    uint8_t *h = q.h + (size_t)env * q.h_env;
    if (r0 < rl) {
      if (SAVE) nm_state_copy(blob + x0, h + r0, rl - r0);
      else nm_state_copy(h + r0, blob + x0, rl - r0);
    }
    if (SAVE && max(r0, live) < r1) nm_state_zero(blob + q.b_off + max(r0, live), r1 - max(r0, live));
  }
}

extern "C" __global__ void __launch_bounds__(NM_STATE_THREADS) nmmo_state_save_kernel(const __grid_constant__ NmStateArgs a, uint8_t *blobs) {
  state_body<true>(a, blobs);
}
extern "C" __global__ void __launch_bounds__(NM_STATE_THREADS) nmmo_state_load_kernel(const __grid_constant__ NmStateArgs a, const uint8_t *blobs) {
  state_body<false>(a, (uint8_t *)blobs);
}
