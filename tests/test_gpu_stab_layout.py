"""Layout of the thread-per-env stabilization process launch (k_stabilize.cu): a full resident grid, 32 queued envs per
warp, warp ranks dealt round the blocks first.  A queue longer than the grid takes further passes; each queued env must
be stabilized exactly once, with the results of a short queue."""
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


def test_long_stabilization_queue_matches_short_one(torch_cuda):
    """65,536 envs: with B200MOBY_STAB_SELECT=0 every env is queued (on a B200 a second pass over the grid), with
    selection only the few that need it (about one warp per SM).  States and every counter must be equal, and the
    process launch must have taken each queued env once."""
    from moby_b200 import TimeSteppingSimulator
    ne, steps = 65536, 120
    sc = scenes.small_lcp_batch(ne, seed=0xB200)
    sc.stabilization_max_iterations = -1
    res = []
    for sel in ("0", "1"):
        os.environ["B200MOBY_STAB_SELECT"] = sel
        try:
            sim = TimeSteppingSimulator(sc)
        finally:
            del os.environ["B200MOBY_STAB_SELECT"]
        sim.kernel_profile(enable=False, reset=True)
        sim.step(1e-3, steps)
        kp = {k["name"]: k for k in sim.kernel_profile(enable=False, reset=True)}
        res.append((sim.counters(), sim.get_state(), kp["stabilize_thread_kernel"]["envs"]))
    assert res[0][0] == res[1][0], (res[0][0], res[1][0])
    assert np.array_equal(res[0][1][0], res[1][1][0]) and np.array_equal(res[0][1][1], res[1][1][1])
    assert res[0][2] == ne * steps, res[0][2]
    assert 0 < res[1][2] < ne * steps and res[0][0]["stab_lcp_solves"] > 0
