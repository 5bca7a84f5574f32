"""ctypes binding of the C ABI (include/nmmo_b200.h) + zero-copy torch views of its buffers.

There is no fallback path: if the CUDA library is missing or no GPU is visible, creating a
simulator raises.
"""
from __future__ import annotations

import ctypes as C
from pathlib import Path
from typing import Optional

import numpy as np

from .config import SPEC

_LIB_PATH = Path(__file__).resolve().parent / "_build" / "libnmmo_b200.so"
_lib = None

EXPORTS = [
    "nmmo_create", "nmmo_destroy", "nmmo_reset", "nmmo_step", "nmmo_step_envs", "nmmo_step_host", "nmmo_step_host_i16", "nmmo_step_host_u8", "nmmo_sample_actions", "nmmo_forage_actions",
    "nmmo_obs_ptr", "nmmo_reward_ptr", "nmmo_terminated_ptr", "nmmo_truncated_ptr", "nmmo_mask_ptr",
    "nmmo_info_ptr", "nmmo_info_valid_ptr", "nmmo_episode_done_ptr", "nmmo_task_id_ptr", "nmmo_task_embed_ptr", "nmmo_obs_stride", "nmmo_num_envs",
    "nmmo_num_agents", "nmmo_step_kernel_name", "nmmo_obs_kernel_name", "nmmo_inject_rng", "nmmo_snapshot", "nmmo_task_state", "nmmo_stats", "nmmo_check", "nmmo_timing", "nmmo_timing_read", "nmmo_profile", "nmmo_set_obs_full", "nmmo_set_autosample",
    "nmmo_state_bytes", "nmmo_save_envs", "nmmo_load_envs", "nmmo_set_event_log", "nmmo_events", "nmmo_last_error",
    "nmmo_rollout_create", "nmmo_rollout_create_compact", "nmmo_rollout_store_compact", "nmmo_rollout_expand", "nmmo_rollout_destroy", "nmmo_rollout_reset", "nmmo_rollout_store", "nmmo_rollout_store_range", "nmmo_rollout_ptr",
    "nmmo_rollout_gae", "nmmo_rollout_buffer", "nmmo_rollout_last_error",
]


class NmmoError(RuntimeError):
    pass


def load(build_if_missing: bool = True):
    """Load libnmmo_b200.so (building it in-tree with nvcc if needed). Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing:
        from . import build as _build
        try:
            _build.build()
        except Exception as e:  # noqa: BLE001
            if not _LIB_PATH.exists():
                raise NmmoError(f"CUDA extension missing and could not be built: {e}") from e
    if not _LIB_PATH.exists():
        raise NmmoError(f"CUDA extension not found at {_LIB_PATH}; run `python -m nmmo_b200.build`")
    import os
    L = C.CDLL(os.environ.get("NMMO_B200_LIB", str(_LIB_PATH)))      # (development: A/B builds of the same ABI)
    vp = C.c_void_p
    L.nmmo_create.restype = C.c_int
    L.nmmo_create.argtypes = [vp, C.c_int, vp, C.c_int, C.c_int, C.c_int, C.c_int, vp, C.c_int, vp, vp, C.c_int, C.POINTER(vp)]
    L.nmmo_destroy.argtypes = [vp]
    L.nmmo_reset.restype = C.c_int
    L.nmmo_reset.argtypes = [vp, vp, vp, vp, vp, vp]
    L.nmmo_step.restype = C.c_int
    L.nmmo_step.argtypes = [vp, vp, vp]
    L.nmmo_step_envs.restype = C.c_int
    L.nmmo_step_envs.argtypes = [vp, C.c_int, C.c_int, vp, vp]
    L.nmmo_step_host.restype = C.c_int
    L.nmmo_step_host.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.nmmo_step_host_i16.restype = C.c_int
    L.nmmo_step_host_i16.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.nmmo_step_host_u8.restype = C.c_int
    L.nmmo_step_host_u8.argtypes = [vp, vp, vp, vp, vp, vp, vp, vp]
    L.nmmo_sample_actions.restype = C.c_int
    L.nmmo_sample_actions.argtypes = [vp, C.c_uint64, vp, vp]
    L.nmmo_forage_actions.restype = C.c_int
    L.nmmo_forage_actions.argtypes = [vp, C.c_uint64, vp, vp]
    for n in ("nmmo_obs_ptr", "nmmo_reward_ptr", "nmmo_terminated_ptr", "nmmo_truncated_ptr", "nmmo_mask_ptr",
              "nmmo_info_ptr", "nmmo_info_valid_ptr", "nmmo_episode_done_ptr", "nmmo_task_id_ptr", "nmmo_task_embed_ptr"):
        getattr(L, n).restype = vp
        getattr(L, n).argtypes = [vp]
    for n in ("nmmo_obs_stride", "nmmo_num_envs", "nmmo_num_agents"):
        getattr(L, n).restype = C.c_int
        getattr(L, n).argtypes = [vp]
    for n in ("nmmo_step_kernel_name", "nmmo_obs_kernel_name"):
        getattr(L, n).restype = C.c_char_p
        getattr(L, n).argtypes = [vp]
    L.nmmo_inject_rng.restype = C.c_int
    L.nmmo_inject_rng.argtypes = [vp, C.c_int, vp, vp, C.c_int]
    L.nmmo_snapshot.restype = C.c_int
    L.nmmo_snapshot.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    L.nmmo_task_state.restype = C.c_int
    L.nmmo_task_state.argtypes = [vp, C.c_int, vp, vp, vp, vp]
    L.nmmo_stats.restype = C.c_int
    L.nmmo_stats.argtypes = [vp, vp, vp, vp, C.c_int]
    L.nmmo_check.restype = C.c_int
    L.nmmo_check.argtypes = [vp]
    L.nmmo_timing.restype = C.c_int
    L.nmmo_timing.argtypes = [vp, C.c_int]
    L.nmmo_timing_read.restype = C.c_int
    L.nmmo_timing_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int)]
    L.nmmo_set_obs_full.restype = C.c_int
    L.nmmo_set_obs_full.argtypes = [vp, C.c_int]
    L.nmmo_set_autosample.restype = C.c_int
    L.nmmo_set_autosample.argtypes = [vp, C.c_uint64, vp]
    L.nmmo_profile.restype = C.c_int
    L.nmmo_profile.argtypes = [vp, C.c_int, vp]
    L.nmmo_state_bytes.restype = C.c_int
    L.nmmo_state_bytes.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.nmmo_save_envs.restype = C.c_int
    L.nmmo_save_envs.argtypes = [vp, vp, C.c_int, vp, vp]
    L.nmmo_load_envs.restype = C.c_int
    L.nmmo_load_envs.argtypes = [vp, vp, C.c_int, vp, vp]
    L.nmmo_set_event_log.restype = C.c_int
    L.nmmo_set_event_log.argtypes = [vp, C.c_int]
    L.nmmo_events.restype = C.c_int
    L.nmmo_events.argtypes = [vp, C.c_int, C.c_int, vp, C.c_int, vp, vp]
    L.nmmo_last_error.restype = C.c_char_p
    L.nmmo_rollout_create.restype = C.c_int
    L.nmmo_rollout_create.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.nmmo_rollout_create_compact.restype = C.c_int
    L.nmmo_rollout_create_compact.argtypes = [C.c_int] * 11 + [C.POINTER(vp)]
    L.nmmo_rollout_store_compact.restype = C.c_int
    L.nmmo_rollout_store_compact.argtypes = [vp] + [vp] * 9 + [C.c_int, vp]
    L.nmmo_rollout_expand.restype = C.c_int
    L.nmmo_rollout_expand.argtypes = [vp, vp, C.c_int, vp, vp, vp]
    L.nmmo_rollout_destroy.argtypes = [vp]
    L.nmmo_rollout_reset.restype = C.c_int
    L.nmmo_rollout_reset.argtypes = [vp, vp]
    L.nmmo_rollout_store.restype = C.c_int
    L.nmmo_rollout_store.argtypes = [vp] + [vp] * 8 + [C.c_int, vp]
    L.nmmo_rollout_store_range.restype = C.c_int
    L.nmmo_rollout_store_range.argtypes = [vp, C.c_int, C.c_int] + [vp] * 9 + [C.c_int, vp]
    L.nmmo_rollout_ptr.restype = C.c_int
    L.nmmo_rollout_ptr.argtypes = [vp, vp, C.POINTER(C.c_int)]
    L.nmmo_rollout_gae.restype = C.c_int
    L.nmmo_rollout_gae.argtypes = [vp, C.c_double, C.c_double, vp]
    L.nmmo_rollout_buffer.restype = vp
    L.nmmo_rollout_buffer.argtypes = [vp, C.c_int]
    L.nmmo_rollout_last_error.restype = C.c_char_p
    _lib = L
    return L


def _p(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class _DevView:
    """Minimal __cuda_array_interface__ holder so torch wraps a handle-owned buffer zero-copy."""

    def __init__(self, ptr: int, shape, typestr: str, owner):
        self.__cuda_array_interface__ = {"shape": tuple(shape), "typestr": typestr, "data": (int(ptr), False),
                                         "version": 2, "strides": None}
        self._owner = owner


def pack_actions_u8(actions, out=None):
    """int actions [..., 12] -> the 12-byte-per-agent format of nmmo_step_host_u8 (include/nmmo_b200.h): byte k = head
    k's index, bits 8.. of Buy.MarketItem (head 2) in bits 2..7 of byte 0.  Works on numpy arrays and torch tensors
    (pack on the device before the copy to the host)."""
    if hasattr(actions, "numpy") and not isinstance(actions, np.ndarray):      # torch tensor
        import torch
        a = actions.to(torch.int32)
        lo = (a & 0xff)
        lo[..., 0] = (a[..., 0] & 3) | (((a[..., 2] >> 8) & 0x3f) << 2)
        res = lo.to(torch.uint8)
        if out is not None:
            out.copy_(res); return out
        return res
    a = np.asarray(actions).astype(np.int32)
    lo = a & 0xff
    lo[..., 0] = (a[..., 0] & 3) | (((a[..., 2] >> 8) & 0x3f) << 2)
    res = lo.astype(np.uint8)
    if out is not None:
        out[...] = res; return out
    return res


class Simulator:
    """Thin object wrapper of one nmmo_handle (one GPU, E environments)."""

    def __init__(self, cfg: np.ndarray, fcfg: np.ndarray, n_envs: int, maps: np.ndarray, task_table: np.ndarray,
                 task_embed: np.ndarray, device: int = 0, env_base: int = 0):
        import torch
        self.torch = torch
        if not torch.cuda.is_available():
            raise NmmoError("no CUDA device visible: nmmo_b200 has no CPU fallback")
        self.L = load()
        self.cfg = np.ascontiguousarray(cfg, np.int32)
        self.fcfg = np.ascontiguousarray(fcfg, np.float64)
        maps = np.ascontiguousarray(maps, np.uint8)
        task_table = np.ascontiguousarray(task_table, np.int32)
        task_embed = np.ascontiguousarray(task_embed, np.uint16)
        S = int(cfg[SPEC["NC_MAP_SIZE"]])
        assert maps.ndim == 3 and maps.shape[1:] == (S, S), "maps must be uint8 [n_maps, S, S]"
        assert task_table.shape[1] == SPEC["NM_TASK_COLS"]
        assert task_embed.shape == (task_table.shape[0], int(cfg[SPEC["NC_TASK_DIM"]]))
        from .tasks import PRED, STATE_PREDICATES
        ok2 = np.array([PRED[n] for n in STATE_PREDICATES])
        bad = task_table[(task_table[:, 7] != 0) & ~np.isin(task_table[:, 5], ok2)]
        if len(bad) or (~np.isin(task_table[:, 7], (0, 1, 2))).any():
            raise NmmoError("combined tasks: combine must be 0/1/2 and the second predicate a state predicate")
        self.device = int(device)
        self.E = int(n_envs)
        self.P = int(cfg[SPEC["NC_N_PLAYERS"]]); self.N = int(cfg[SPEC["NC_N_NPCS"]])
        self.cap = int(cfg[SPEC["NC_ITEM_CAP"]]); self.S = S
        h = C.c_void_p()
        rc = self.L.nmmo_create(_p(self.cfg), len(self.cfg), _p(self.fcfg), len(self.fcfg), self.E, self.device,
                                int(env_base), _p(maps), maps.shape[0], _p(task_table), _p(task_embed),
                                task_table.shape[0], C.byref(h))
        self._check(rc)
        self.h = h
        self.stride = self.L.nmmo_obs_stride(self.h)
        n = self.E * self.P
        dev = torch.device("cuda", self.device)

        def view(fn, shape, typestr):
            ptr = getattr(self.L, fn)(self.h)
            return torch.as_tensor(_DevView(ptr, shape, typestr, self), device=dev)

        with torch.cuda.device(dev):
            self.obs = view("nmmo_obs_ptr", (n, self.stride), "|u1")
            self.rewards = view("nmmo_reward_ptr", (n,), "<f4")
            self.terminated = view("nmmo_terminated_ptr", (n,), "|u1")
            self.truncated = view("nmmo_truncated_ptr", (n,), "|u1")
            self.mask = view("nmmo_mask_ptr", (n,), "|u1")
            self.info = view("nmmo_info_ptr", (n, SPEC["IN_N"]), "<f4")
            self.info_valid = view("nmmo_info_valid_ptr", (n,), "|u1")
            self.episode_done = view("nmmo_episode_done_ptr", (self.E,), "|u1")
            self.task_id = view("nmmo_task_id_ptr", (n,), "<i4")
            self.task_embed_ptr = self.L.nmmo_task_embed_ptr(self.h)
            self.actions = torch.zeros((self.E, self.P, 12), dtype=torch.int32, device=dev)
        nb = C.c_size_t()
        self._check(self.L.nmmo_state_bytes(self.h, C.byref(nb)))
        self.state_bytes = int(nb.value)      # bytes of one environment's saved state (save_envs / load_envs)

    def _check(self, rc: int):
        if rc != 0:
            raise NmmoError(f"nmmo_b200 error {rc}: {self.L.nmmo_last_error().decode()}")

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "h", None):
            self.L.nmmo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def reset(self, seeds, map_ids=None, task_ids=None, env_mask=None):
        seeds = np.ascontiguousarray(np.broadcast_to(np.asarray(seeds, np.uint64), (self.E,)))
        m = None if map_ids is None else np.ascontiguousarray(map_ids, np.int32).reshape(self.E)
        t = None if task_ids is None else np.ascontiguousarray(task_ids, np.int32).reshape(self.E, self.P)
        k = None if env_mask is None else np.ascontiguousarray(env_mask, np.uint8).reshape(self.E)
        self._check(self.L.nmmo_reset(self.h, _p(seeds), _p(m), _p(t), _p(k), self._stream()))

    def step(self, actions=None):
        """actions: int32 CUDA tensor [E, P, 12] (defaults to self.actions). Asynchronous."""
        a = self.actions if actions is None else actions
        assert a.is_cuda and a.dtype == self.torch.int32 and a.is_contiguous() and a.numel() == self.E * self.P * 12
        self._check(self.L.nmmo_step(self.h, C.c_void_p(a.data_ptr()), self._stream()))

    def step_envs(self, lo: int, hi: int, actions):
        """Step envs [lo, hi) only: actions int32 CUDA tensor [hi - lo, P, 12] (row 0 = env lo). Asynchronous; ranges
        stepped on different streams may overlap in time when they are disjoint."""
        a = actions
        assert a.is_cuda and a.dtype == self.torch.int32 and a.is_contiguous()
        if a.numel() != max(int(hi) - int(lo), 0) * self.P * 12:
            raise ValueError(f"actions of envs [{lo}, {hi}) must hold {(hi - lo) * self.P * 12} values, got {a.numel()}")
        self._check(self.L.nmmo_step_envs(self.h, int(lo), int(hi), C.c_void_p(a.data_ptr()), self._stream()))

    def save_envs(self, env_ids, out=None):
        """Saved state of envs `env_ids` (duplicates allowed) -> uint8 CUDA tensor [n, state_bytes] on this handle's device
        (or `out`, a contiguous uint8 tensor of that shape there).  Asynchronous on the current stream.  torch.save of the
        tensor is a checkpoint of those envs (DESIGN.md 2.3)."""
        ids = np.ascontiguousarray(np.asarray(env_ids, np.int64).reshape(-1), np.int32)
        t = self.torch
        if out is None:
            out = t.empty((len(ids), self.state_bytes), dtype=t.uint8, device=t.device("cuda", self.device))
        if not (out.is_cuda and out.device.index == self.device and out.dtype == t.uint8 and out.is_contiguous()
                and tuple(out.shape) == (len(ids), self.state_bytes)):
            raise ValueError(f"out must be a contiguous uint8 tensor [{len(ids)}, {self.state_bytes}] on cuda:{self.device}")
        self._check(self.L.nmmo_save_envs(self.h, _p(ids), len(ids), C.c_void_p(out.data_ptr()), self._stream()))
        return out

    def load_envs(self, env_ids, states):
        """Load states[i] (a row of save_envs, from this or another handle of the same world and family) into env
        env_ids[i]; a CPU tensor, e.g. one read back with torch.load, is copied to the device first.  The loaded envs'
        observations, masks, outputs and built-in-policy rows become those of the tick they were saved at; their next
        step continues the saved episode."""
        ids = np.ascontiguousarray(np.asarray(env_ids, np.int64).reshape(-1), np.int32)
        t = self.torch
        s = states if t.is_tensor(states) else t.as_tensor(np.asarray(states))
        if s.dtype != t.uint8 or tuple(s.shape) != (len(ids), self.state_bytes):
            raise ValueError(f"states must be uint8 [{len(ids)}, {self.state_bytes}], got {s.dtype} {tuple(s.shape)}")
        s = s.to(device=t.device("cuda", self.device), non_blocking=False).contiguous()
        self._check(self.L.nmmo_load_envs(self.h, _p(ids), len(ids), C.c_void_p(s.data_ptr()), self._stream()))

    def set_event_log(self, enable: bool = True):
        """Event log on (allocates E * ring size * 8 bytes of device staging, zeroes every env's events) or off (frees
        it).  While it is on, every step keeps the player events each stepped env emitted; events() hands them out."""
        self._check(self.L.nmmo_set_event_log(self.h, int(bool(enable))))

    def events(self, lo: int = 0, hi: Optional[int] = None, out=None, count=None):
        """The last step's events of envs [lo, hi) (default all) -> (rows int32 CUDA [cap, 9], count int32 CUDA [1]).
        A row is [env, ent_id, tick, event, type, level, number, gold, target] (columns 1..8 as in the reference's event
        log; env is the handle's env index), ordered by env, agent, then the order the agent's events happened in.
        count[0] is the number of rows of the range; only the first cap = len(out) of them are written (without `out`,
        cap = (hi - lo) * max(8 * P, 1024)).  Asynchronous on the current stream: nothing is read back to the host."""
        t = self.torch
        hi = self.E if hi is None else int(hi)
        dev = t.device("cuda", self.device)
        if out is None:
            out = t.empty((max(hi - int(lo), 0) * max(8 * self.P, 1024), 9), dtype=t.int32, device=dev)
        if count is None:
            count = t.empty(1, dtype=t.int32, device=dev)
        for name, x, shape in (("out", out, (out.shape[0], 9)), ("count", count, (1,))):
            if not (x.is_cuda and x.device.index == self.device and x.dtype == t.int32 and x.is_contiguous() and tuple(x.shape) == shape):
                raise ValueError(f"{name} must be a contiguous int32 tensor {list(shape)} on cuda:{self.device}")
        self._check(self.L.nmmo_events(self.h, int(lo), hi, C.c_void_p(out.data_ptr()), int(out.shape[0]),
                                       C.c_void_p(count.data_ptr()), self._stream()))
        return out, count

    def step_host(self, actions: np.ndarray, want_obs: bool = False):
        """Host-buffer call: actions [E,P,12] in host memory (pinned = async copies) as int32, int16 (half the
        bytes over the host link) or uint8 packed by ``pack_actions_u8`` (a quarter)."""
        dt = getattr(actions, "dtype", None)
        i16, u8 = dt == np.int16, dt == np.uint8
        a = np.ascontiguousarray(actions, np.uint8 if u8 else (np.int16 if i16 else np.int32)).reshape(self.E, self.P, 12)
        n = self.E * self.P
        if getattr(self, "_host_out", None) is None:
            t = self.torch
            self._host_out = (t.empty(n, dtype=t.float32).pin_memory(), t.empty(n, dtype=t.uint8).pin_memory(),
                              t.empty(n, dtype=t.uint8).pin_memory(), t.empty(n, dtype=t.uint8).pin_memory())
            # numpy views and C pointers of the pinned result buffers, made once (this call sits on an idle GPU: a
            # host-buffer step ends in a stream synchronise, so every microsecond of Python before the first copy counts)
            self._host_out_np = tuple(x.numpy() for x in self._host_out)
            self._host_out_p = tuple(_p(x) for x in self._host_out_np)
        rew, term, trunc, mask = self._host_out_np
        obs = np.empty((n, self.stride), np.uint8) if want_obs else None
        fn = self.L.nmmo_step_host_u8 if u8 else (self.L.nmmo_step_host_i16 if i16 else self.L.nmmo_step_host)
        self._check(fn(self.h, _p(a), *self._host_out_p, _p(obs), self._stream()))
        return rew, term, trunc, mask, obs

    def sample_actions(self, seed: int, out=None):
        a = self.actions if out is None else out
        self._check(self.L.nmmo_sample_actions(self.h, C.c_uint64(int(seed)), C.c_void_p(a.data_ptr()), self._stream()))
        return a

    def forage_actions(self, seed: int, out=None):
        """Scripted survival policy (nmmo_forage_actions): walk to the nearest water / foliage when hungry, else explore."""
        a = self.actions if out is None else out
        self._check(self.L.nmmo_forage_actions(self.h, C.c_uint64(int(seed)), C.c_void_p(a.data_ptr()), self._stream()))
        return a

    def inject_rng(self, env: int, keys, vals):
        k = np.ascontiguousarray(keys, np.uint64); v = np.ascontiguousarray(vals, np.uint32)
        self._check(self.L.nmmo_inject_rng(self.h, int(env), _p(k), _p(v), len(k)))

    def snapshot(self, env: int):
        ent = np.zeros((self.P + self.N, SPEC["EA_N"]), np.int16)
        items = np.zeros((self.cap, SPEC["IS_N"]), np.int16)
        mp = np.zeros((self.S, self.S), np.uint8)
        sc = np.zeros(16, np.int32)
        self._check(self.L.nmmo_snapshot(self.h, int(env), _p(ent), _p(items), _p(mp), _p(sc)))
        return ent, items, mp, sc

    def task_state(self, env: int):
        """(task_id, completed tick, reward_signal_count, max_progress) of one env's agents (stat_wrapper.py:155-159)."""
        tid = np.zeros(self.P, np.int32); comp = np.zeros(self.P, np.int32); sig = np.zeros(self.P, np.int32)
        mp = np.zeros(self.P, np.float64)
        self._check(self.L.nmmo_task_state(self.h, int(env), _p(tid), _p(comp), _p(sig), _p(mp)))
        return tid, comp, sig, mp

    def stats(self, clear: bool = False):
        sums = np.zeros(SPEC["IN_N"], np.float64); counts = np.zeros(SPEC["IN_N"], np.float64)
        counters = np.zeros(8, np.uint64)
        self._check(self.L.nmmo_stats(self.h, _p(sums), _p(counts), _p(counters), int(clear)))
        return sums, counts, counters

    def kernel_names(self):
        """(step kernel, observation kernel) instantiations this handle launches."""
        return self.L.nmmo_step_kernel_name(self.h).decode(), self.L.nmmo_obs_kernel_name(self.h).decode()

    def check(self):
        """Raises NmmoError if any environment dropped events (event ring overflow) since the last stats clear."""
        self._check(self.L.nmmo_check(self.h))

    def timing(self, enable: bool):
        self._check(self.L.nmmo_timing(self.h, int(enable)))

    def timing_read(self):
        a, b, n = C.c_double(), C.c_double(), C.c_int()
        self._check(self.L.nmmo_timing_read(self.h, C.byref(a), C.byref(b), C.byref(n)))
        return a.value, b.value, n.value

    def profile(self, enable: bool):
        out = np.zeros(64, np.uint64)
        self._check(self.L.nmmo_profile(self.h, int(enable), _p(out)))
        return out

    def set_obs_full(self, full: bool):
        self._check(self.L.nmmo_set_obs_full(self.h, int(full)))

    def set_autosample(self, seed, out=None, enable: bool = True):
        """Built-in random policy: every observation pass also writes uniform-random valid actions
        into `out` (default self.actions)."""
        a = self.actions if out is None else out
        ptr = C.c_void_p(a.data_ptr()) if enable else None
        self._check(self.L.nmmo_set_autosample(self.h, C.c_uint64(int(seed)), ptr))
