"""CPU check of the first-rung hand-off of the one-thread group (sim_device.cuh: EnvCtx::first_rung): under a budget an
env whose first lcp_fast rung does not verify is abandoned untouched and re-solved by the straggler phase.  With a
budget too large to run out, only that hand-off moves envs; the phased schedule must still give the fused loop's bits."""
import numpy as np
import pytest

from moby_b200 import scenes


@pytest.fixture(scope="module")
def hostsim():
    import hostsim_api
    hostsim_api.build()
    return hostsim_api


def test_first_rung_handoff_matches_fused(hostsim):
    sc = scenes.small_lcp_batch(64, seed=11)
    a, b = hostsim.HostSim(sc), hostsim.HostSim(sc)
    a.step(1e-3, 80)
    for _ in range(8):
        b.step_phased(1e-3, 10, rounds=2, pivot_budget=1 << 20)
    assert np.array_equal(a.q, b.q) and np.array_equal(a.v, b.v) and np.array_equal(a.time, b.time)
    assert np.array_equal(a.zlast_n, b.zlast_n)
    for e in range(64):
        assert np.array_equal(a.zlast[:a.zlast_n[e], e], b.zlast[:b.zlast_n[e], e])
    ca, cb = a.counters_dict(), b.counters_dict()
    assert ca["lcp_solves"] > 100 and ca["lcp_fast_calls"] > ca["lcp_solves"]   # some first rungs did not verify
    assert ca == cb, (ca, cb)
