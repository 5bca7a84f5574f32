"""Device-resident rollout storage + GAE behind the names the reference trainer uses.

Mirrors the storage part of ``clean_pufferl`` (/root/reference/reinforcement_learning/clean_pufferl.py):
the ``obs / actions / logprobs / rewards / dones / values`` arrays of ``batch_size + 1`` rows (:183-197),
the masked append of one ``recv()`` with its ``sort_keys`` (:329-348), the sort by ``(env_id, step)``
(:413-414) and the GAE loop (:424-436) -- but every buffer lives in HBM and the work is done by the CUDA
kernels of csrc/nmmo_rollout.cu through the C ABI (include/nmmo_b200.h, ``nmmo_rollout_*``).  There is no
CPU fallback: constructing a DeviceRollout without the CUDA library or a GPU raises.
"""
from __future__ import annotations

import ctypes as C

from .lib import NmmoError, _DevView, load

_BUF = {"obs": 0, "actions": 1, "logprobs": 2, "rewards": 3, "dones": 4, "values": 5, "slot": 6, "step": 7,
        "idxs": 8, "advantages": 9}


class DeviceRollout:
    """compact = a dict(agents_per_env, market_off, market_bytes, task_off, task_bytes, max_steps, task_embed_ptr) -- see
    ``DeviceRollout.compact_for(sim)`` -- stores the Market block once per (step, env) and the Task block as the task id
    (a row shrinks from 25 344 to 8 960 bytes); ``expand(idxs)`` re-assembles whole records for a minibatch."""

    @staticmethod
    def compact_for(sim, max_steps: int = 64) -> dict:
        from .config import ObsLayout
        L = ObsLayout(sim.cfg)
        return dict(agents_per_env=sim.P, market_off=L.o_market, market_bytes=L.n_mkt * 32, task_off=L.o_task,
                    task_bytes=L.task_dim * 2, ids_off=L.o_ids, max_steps=int(max_steps), task_embed_ptr=sim.task_embed_ptr)

    def __init__(self, batch_size: int, n_slots: int, obs_stride: int, device: int = 0, compact: dict = None):
        import torch
        self.torch = torch
        if not torch.cuda.is_available():
            raise NmmoError("no CUDA device visible: nmmo_b200 has no CPU fallback")
        self.L = load()
        self.batch_size, self.n_slots, self.obs_stride, self.device = int(batch_size), int(n_slots), int(obs_stride), int(device)
        h = C.c_void_p()
        self.compact = compact
        if compact:
            self._check(self.L.nmmo_rollout_create_compact(self.device, self.batch_size, self.n_slots, self.obs_stride,
                                                           compact["agents_per_env"], compact["market_off"], compact["market_bytes"],
                                                           compact["task_off"], compact["task_bytes"], compact["ids_off"], compact["max_steps"], C.byref(h)))
            self.row_stride = self.obs_stride - compact["market_bytes"] - compact["task_bytes"]
        else:
            self._check(self.L.nmmo_rollout_create(self.device, self.batch_size, self.n_slots, self.obs_stride, C.byref(h)))
            self.row_stride = self.obs_stride
        self.h = h
        dev = torch.device("cuda", self.device)
        rows = self.batch_size + 1

        def view(name, shape, typestr):
            ptr = self.L.nmmo_rollout_buffer(self.h, _BUF[name])
            return torch.as_tensor(_DevView(ptr, shape, typestr, self), device=dev)

        with torch.cuda.device(dev):
            self.obs = view("obs", (rows, self.row_stride), "|u1")
            self.actions = view("actions", (rows, 12), "<i4")
            self.logprobs = view("logprobs", (rows,), "<f4")
            self.rewards = view("rewards", (rows,), "<f4")
            self.dones = view("dones", (rows,), "<f4")
            self.values = view("values", (rows,), "<f4")
            self.slot = view("slot", (rows,), "<i4")
            self.step = view("step", (rows,), "<i4")
            self.idxs = view("idxs", (rows,), "<i4")
            self.advantages = view("advantages", (rows,), "<f4")
        self.reset()

    def _check(self, rc: int):
        if rc != 0:
            raise NmmoError(f"nmmo_b200 rollout error {rc}: {self.L.nmmo_rollout_last_error().decode()}")

    def _stream(self):
        return C.c_void_p(self.torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "h", None):
            self.L.nmmo_rollout_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass

    def reset(self):
        self._check(self.L.nmmo_rollout_reset(self.h, self._stream()))

    def _dev(self, t, dtype):
        t = t if self.torch.is_tensor(t) else self.torch.as_tensor(t)
        return t.to(device=self.obs.device, dtype=dtype).contiguous()

    def store(self, o, value, actions, logprob, r, d, mask, step: int, learner_mask=None, task_id=None, slot_base: int = 0):
        """Append one ``recv()`` (clean_pufferl.py:329-348); every argument is (or becomes) a CUDA tensor.  A compact
        rollout also needs ``task_id`` (``sim.task_id``: int32 [n_slots] on the device).

        The arguments cover ``len(mask)`` slots starting at ``slot_base``: a ``recv()`` of an env pool hands out one batch,
        whose rows are the global agent slots ``[slot_base, slot_base + len(mask))`` (``slot_base = lo * agents_per_env``
        for ``pool.batch_env_range == (lo, hi)``); the sort key is the global slot.  ``task_id`` is then the batch's slice."""
        t = self.torch
        mask = self._dev(mask, t.uint8).reshape(-1)
        n = mask.numel()
        o = self._dev(o, t.uint8); actions = self._dev(actions, t.int32).reshape(n, 12)
        value = self._dev(value, t.float32).reshape(-1); logprob = self._dev(logprob, t.float32).reshape(-1)
        r = self._dev(r, t.float32).reshape(-1); d = self._dev(d, t.float32).reshape(-1)
        lm = None if learner_mask is None else self._dev(learner_mask, t.uint8).reshape(-1)
        for x in (value, logprob, r, d, lm):
            if x is not None and x.numel() != n:
                raise ValueError(f"store(): every per-slot argument must hold len(mask) = {n} entries")
        if o.shape[0] != n:
            raise ValueError(f"store(): obs must hold len(mask) = {n} records")
        p = lambda x: None if x is None else C.c_void_p(x.data_ptr())  # noqa: E731
        tid = None
        if self.compact:
            if task_id is None:
                raise NmmoError("compact rollout: store() needs task_id (Simulator.task_id)")
            tid = self._dev(task_id, t.int32).reshape(-1)
            if tid.numel() != n:
                raise ValueError(f"store(): task_id must hold len(mask) = {n} entries")
        self._check(self.L.nmmo_rollout_store_range(self.h, int(slot_base), n, p(o), p(actions), p(logprob), p(value), p(r), p(d),
                                                    p(mask), p(lm), p(tid), int(step), self._stream()))

    def expand(self, idxs=None, n: int = None, out=None):
        """Whole observation records of rows ``idxs`` (int32 CUDA tensor; None = rows 0..n-1): the minibatch gather of
        clean_pufferl.py:439-443.  Plain rollouts index ``obs`` directly; compact ones re-assemble Market and Task."""
        t = self.torch
        if idxs is not None:
            idxs = self._dev(idxs, t.int32).reshape(-1)
            n = idxs.numel()
        if not self.compact:
            return self.obs[:n] if idxs is None else self.obs[idxs.long()]
        if out is None:
            out = t.empty((n, self.obs_stride), dtype=t.uint8, device=self.obs.device)
        self._check(self.L.nmmo_rollout_expand(self.h, None if idxs is None else C.c_void_p(idxs.data_ptr()), int(n),
                                               C.c_void_p(self.compact["task_embed_ptr"]), C.c_void_p(out.data_ptr()), self._stream()))
        return out

    @property
    def ptr(self) -> int:
        v = C.c_int(0)
        self._check(self.L.nmmo_rollout_ptr(self.h, self._stream(), C.byref(v)))
        return v.value

    def gae(self, gamma: float, gae_lambda: float):
        """Sorted order (``idxs``) and ``advantages`` of the stored rows (clean_pufferl.py:413-436)."""
        self._check(self.L.nmmo_rollout_gae(self.h, float(gamma), float(gae_lambda), self._stream()))
        return self.idxs, self.advantages
