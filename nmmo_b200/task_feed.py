"""Host curricula at automatic resets: keep one pending next-episode task per env of a B200VecEnv.

The reference's ``--syllabus`` run (syllabus_wrapper.py:20-33,73-207) hands every reset a task from its curriculum and
tells the curriculum how each episode went.  On this backend an env resets itself inside the step call after its
episode ends, so the task has to be on the device before that step: ``TaskFeed`` keeps exactly one pending task per env
(``B200VecEnv.set_next_episodes``), reports each finished episode with the task it ran, and refills the env's entry once
the reset that consumed it has been issued.

When that is depends on how the pool reports finishes.  With ``collect_infos=True`` a finish is reported by the recv()
whose outputs end the episode, one tick BEFORE the send() that resets the env; with ``collect_infos="async"`` it is
reported one recv() later, AFTER that send().  In an env pool the send() that resets an env is its batch's, and entries
can only be written while the env's batch is the one recv() returned.  So a finished env is queued on its batch and
refilled at the first recv() of that batch after its reset was issued: the same recv() in lock-step "async" mode, the
next recv() of the batch otherwise.  Either way the entry is in place before the new episode can end.

Usage::

    feed = TaskFeed(pool, sample=curriculum_sample, update=curriculum_update)
    feed.start(seed)
    while training:
        obs, rew, term, trunc, infos, env_id, mask = feed.recv()
        feed.send(policy(obs))
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import numpy as np


class TaskFeed:
    """Drives a ``B200VecEnv``'s recv()/send() loop so that every episode of every env runs a task from ``sample``.

    sample(k) -> k task-table rows (ints in [0, n_tasks)).
    update(env, task, infos): called once for each finished episode, with the pool's env index, the task row the episode
    ran and the info dicts of its agents (every agent's end-of-episode record, in the order the pool handed them out).
    """

    def __init__(self, pool, sample: Callable[[int], "np.ndarray"], update: Optional[Callable[[int, int, List[Dict]], None]] = None):
        if pool.collect_infos not in (True, "async"):
            raise ValueError('TaskFeed reads finished episodes from the infos: create the pool with collect_infos=True or "async"')
        self.pool, self.sample, self.update = pool, sample, update
        E = pool.num_envs
        self.running = np.full(E, -1, np.int64)       # task of each env's current episode
        self.pending = np.full(E, -1, np.int64)       # task written for its next episode (-1: consumed, not yet refilled)
        self._infos: List[List[Dict]] = [[] for _ in range(E)]
        self._queue: List[List[int]] = [[] for _ in range(pool.num_batches)]     # per batch: envs to refill at its next recv()

    def _draw(self, k: int) -> np.ndarray:
        rows = np.asarray(self.sample(k), np.int64).reshape(-1)
        if rows.shape != (k,):
            raise ValueError(f"sample({k}) returned {rows.shape[0]} rows")
        return rows

    def start(self, seed: int = 0):
        """Reset every env with a sampled task and give each a sampled task for its next episode."""
        from .dist import global_seeds
        p = self.pool
        E = p.num_envs
        envs = np.arange(E)
        self.running[:] = self._draw(E)
        p.reset_envs(envs, global_seeds(int(seed), p.env_base, E), new_tasks=self.running)
        if p.collect_infos == "async":
            p.drain_infos()                       # records of episodes the reset cut are not this feed's
        self.pending[:] = self._draw(E)
        p.set_next_episodes(envs, tasks=self.pending)
        for q in self._queue:
            q.clear()
        for x in self._infos:
            x.clear()

    def _refill(self, batch: int):
        envs = self._queue[batch]
        if envs:
            rows = self._draw(len(envs))
            self.pending[envs] = rows
            self.pool.set_next_episodes(np.asarray(envs), tasks=rows)
            envs.clear()

    def _finished(self, infos: List[Dict]) -> List[int]:
        """Collect this recv()'s infos per env; the envs whose episode they end."""
        p = self.pool
        done = []
        for slot, info in zip(p.last_info_slots, infos):
            e = int(slot) // p.agents_per_env
            self._infos[e].append(info)
            body = info[p.stat_prefix] if p.stat_prefix else info
            if body.get("episode_done"):
                done.append(e)
        for e in done:
            if self.update is not None:
                self.update(e, int(self.running[e]), self._infos[e])
            self._infos[e] = []
            self.running[e] = self.pending[e]     # the automatic reset takes (or took) the pending task
            self.pending[e] = -1
        return done

    def recv(self):
        """pool.recv(), with the finished episodes reported and the consumed entries refilled."""
        p = self.pool
        out = p.recv()
        k = p.batch_env_range[0] // p.envs_per_batch
        if p.collect_infos == "async":
            # finishes of the batch received before this one: its send() has issued their resets
            for e in self._finished(out[4]):
                self._queue[e // p.envs_per_batch].append(e)
            self._refill(k)
        else:
            # this batch's finishes: their resets are the coming send(); refill at the batch's next recv()
            self._refill(k)
            self._queue[k].extend(self._finished(out[4]))
        return out

    def send(self, actions):
        self.pool.send(actions)
