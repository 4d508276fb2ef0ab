"""First-rung hand-off of the thread-per-env impact classes (sim_device.cuh: EnvCtx::first_rung): an env whose first
lcp_fast rung does not verify is abandoned untouched and re-solved from scratch by the hard-queue launch.  Which kernel
solves an env may change, what it computes may not."""
import os

import numpy as np
import pytest

from moby_b200 import scenes

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    return torch


def _run(sc, steps, handoff):
    from moby_b200 import TimeSteppingSimulator
    os.environ["B200MOBY_FIRST_RUNG_HANDOFF"] = handoff
    try:
        sim = TimeSteppingSimulator(sc)
    finally:
        del os.environ["B200MOBY_FIRST_RUNG_HANDOFF"]
    sim.kernel_profile(enable=False, reset=True)
    sim.step(1e-3, steps)
    kp = {k["name"]: k["envs"] for k in sim.kernel_profile(enable=False, reset=True)}
    return sim.counters(), sim.get_state(), kp["impact_warp_kernel[hard queue]"] + kp["impact_warp_kernel[stragglers]"]


def test_first_rung_handoff_gives_the_same_results(torch_cuda):
    """65,536 envs of the default workload with the hand-off on and off: states and every counter must be equal, and the
    hand-off must really have moved envs to the warp-per-env launches."""
    sc = scenes.small_lcp_batch(65536, seed=0xB200)
    sc.stabilization_max_iterations = -1
    on, off = _run(sc, 120, "1"), _run(sc, 120, "0")
    assert on[0] == off[0], (on[0], off[0])
    assert np.array_equal(on[1][0], off[1][0]) and np.array_equal(on[1][1], off[1][1])
    assert on[0]["lcp_failures"] == 0 and on[0]["lcp_solves"] > 0
    assert on[2] > off[2], (on[2], off[2])
