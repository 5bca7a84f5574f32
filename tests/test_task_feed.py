"""TaskFeed's bookkeeping on a host stand-in for B200VecEnv that keeps its reporting order: an env whose step ends its
episode resets on its batch's next send(), taking the pending task (or a drawn one, -1, when nothing is pending);
collect_infos=True reports the finish in the recv() whose outputs end the episode, "async" one recv() later."""
import numpy as np
import pytest

from nmmo_b200.task_feed import TaskFeed


class FakePool:
    agents_per_env = 2
    stat_prefix = None
    env_base = 0

    def __init__(self, E, b, collect_infos):
        self.num_envs, self.envs_per_batch, self.num_batches = E, b, E // b
        self.collect_infos = collect_infos
        self.lengths = 3 + np.arange(E) % 4            # episode lengths differ per env
        self.task, self.tick = np.zeros(E, int), np.zeros(E, int)
        self.done = np.zeros(E, bool)
        self.flag, self.value = np.zeros(E, bool), np.zeros(E, int)
        self.ran = {e: [] for e in range(E)}           # task of every episode each env started
        self.k, self.idle, self.q = 0, True, []
        self.batch_env_range, self.last_info_slots = (0, b), []

    def reset_envs(self, envs, seeds, new_tasks=None):
        for e, t in zip(envs, new_tasks):
            self.task[e], self.tick[e], self.done[e] = t, 0, False
            self.ran[e].append(int(t))
        self.idle = True

    def drain_infos(self):
        self.q = []
        return []

    def set_next_episodes(self, envs, tasks=None):
        lo, hi = self.batch_env_range
        for e in envs:
            assert self.idle or lo <= e < hi, "entry for an env outside the batch"
        self.flag[envs], self.value[envs] = True, tasks

    def _infos(self, lo, hi):
        slots, infos = [], []
        for e in range(lo, hi):
            if self.done[e]:
                for p in range(self.agents_per_env):
                    slots.append(e * self.agents_per_env + p)
                    info = {"curriculum": {f"task_{self.task[e]}": (0.0, 0)}}
                    if p == self.agents_per_env - 1:
                        info["episode_done"] = True
                    infos.append(info)
        return slots, infos

    def recv(self):
        lo, hi = self.k * self.envs_per_batch, (self.k + 1) * self.envs_per_batch
        self.batch_env_range = (lo, hi)
        now = self._infos(lo, hi)
        if self.collect_infos == "async":
            (self.last_info_slots, infos), self.q = (self.q or ([], [])), now
        else:
            self.last_info_slots, infos = now
        return None, None, None, None, infos, None, None

    def send(self, actions):
        lo, hi = self.batch_env_range
        for e in range(lo, hi):
            if self.done[e]:                            # the automatic reset
                self.task[e] = self.value[e] if self.flag[e] else -1
                self.flag[e], self.tick[e], self.done[e] = False, 0, False
                self.ran[e].append(int(self.task[e]))
            else:
                self.tick[e] += 1
                self.done[e] = self.tick[e] == self.lengths[e]
        self.idle = False
        self.k = (self.k + 1) % self.num_batches


@pytest.mark.parametrize("collect_infos", ["async", True])
@pytest.mark.parametrize("b", [6, 3, 2])
def test_every_reset_takes_the_next_sampled_task(collect_infos, b):
    pool = FakePool(6, b, collect_infos)
    counter = [0]

    def sample(k):
        counter[0] += k
        return np.arange(counter[0] - k, counter[0])

    reported = {e: [] for e in range(6)}

    def update(env, task, infos):
        assert len(infos) == pool.agents_per_env
        assert all(next(iter(i["curriculum"])) == f"task_{task}" for i in infos)
        reported[env].append(task)

    feed = TaskFeed(pool, sample, update)
    feed.start(0)
    for _ in range(100 * pool.num_batches):
        feed.recv()
        feed.send(None)
    tasks = sorted(t for e in range(6) for t in pool.ran[e])
    assert -1 not in tasks, "an automatic reset found no pending task"
    assert len(set(tasks)) == len(tasks), "a sampled task ran twice"
    for e in range(6):
        n = len(reported[e])
        assert n >= 10 and reported[e] == pool.ran[e][:n], (e, reported[e], pool.ran[e])
        assert len(pool.ran[e]) - n <= 2


def test_rejects_pools_without_infos():
    with pytest.raises(ValueError, match="collect_infos"):
        TaskFeed(FakePool(2, 2, False), lambda k: np.zeros(k, int))
