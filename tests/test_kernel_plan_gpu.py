"""GPU: the step and observation kernels a handle launches are the ones kernel_names() reports.  One reset and one step
run under torch.profiler for every kernel the launch plan can choose (both families, four / three / two / one envs per
CTA, the *_std instantiations and the generic ones), and with the phase profiler on or draws injected, which switch the
handle to the generic instantiations."""
import functools

import numpy as np
import pytest

from bench import world
from util import SMALL, build_world

pytestmark = pytest.mark.gpu


@functools.lru_cache(maxsize=None)
def _default():
    return world(n_maps=2)


@functools.lru_cache(maxsize=None)
def _small():
    return build_world(task_dim=64, **SMALL)


@functools.lru_cache(maxsize=None)
def _config5():
    return world(workload="config5", n_maps=2)


NO_STD = {"NMMO_B200_NO_STD_STEP": "1", "NMMO_B200_NO_STD_OBS": "1"}
# case: (world, test hooks, handle mode, envs, the names the handle must report)
CASES = {
    "default": (_default, {}, None, 5, ("nmmo_step4_std_kernel", "nmmo_obs_std_kernel")),
    "no_std": (_default, NO_STD, None, 5, ("nmmo_step4_kernel", "nmmo_obs_kernel")),
    "three_per_cta": (_default, {"NMMO_B200_ENVS_PER_CTA": "3"}, None, 5, ("nmmo_step3_std_kernel", "nmmo_obs_std_kernel")),
    "two_per_cta": (_default, {"NMMO_B200_ENVS_PER_CTA": "2"}, None, 5, ("nmmo_step_kernel", "nmmo_obs_std_kernel")),
    "one_per_cta": (_default, {"NMMO_B200_ENVS_PER_CTA": "1"}, None, 5, ("nmmo_step_kernel", "nmmo_obs_std_kernel")),
    "force_big": (_small, {"NMMO_B200_FORCE_BIG": "1"}, None, 5, ("nmmo_step_big_kernel", "nmmo_obs_big_kernel")),
    "config5": (_config5, {}, None, 2, ("nmmo_step_big_std_kernel", "nmmo_obs_big_std_kernel")),
    "phase_profiler": (_default, {}, "profile", 5, ("nmmo_step4_kernel", "nmmo_obs_kernel")),
    "injected_draws": (_default, {}, "inject", 5, ("nmmo_step4_kernel", "nmmo_obs_std_kernel")),
}


def _launched(sim):
    """The nmmo_step* / nmmo_obs* kernels one reset and one step run, by name, from a CUDA activity trace."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        sim.reset(np.arange(sim.E, dtype=np.uint64) + 1)
        sim.sample_actions(1)
        sim.step()
        torch.cuda.synchronize()
    return {e.name for e in prof.events() if e.name.startswith(("nmmo_step", "nmmo_obs"))}


@pytest.mark.parametrize("case", list(CASES))
def test_launched_kernels_are_the_reported_ones(monkeypatch, case):
    from nmmo_b200.lib import Simulator
    make, hooks, mode, E, expected = CASES[case]
    for k, v in hooks.items():
        monkeypatch.setenv(k, v)
    cfg, fcfg, maps, tab, emb = make()
    sim = Simulator(cfg, fcfg, E, maps, tab, emb)
    try:
        if mode == "profile":
            sim.profile(True)
        elif mode == "inject":
            sim.inject_rng(0, [1], [0])
        assert sim.kernel_names() == expected
        assert _launched(sim) == set(expected)
        assert sim.kernel_names() == expected
    finally:
        sim.close()
