"""example/contact-constrained-pendulum: a pin joint emulated by six frictionless contacts that the scene's collision-detection
plugin generates every step (contact-constrained-pendulum-coldet-plugin.cpp:60-110), here the shapes SHAPE_PIN / SHAPE_PINWORLD.
Every solve is a degenerate 48-variable QP-LCP (three pairs of opposite normals at one point), followed by up to 25
stabilization iterations (the scene's constraint-stabilization-max-iterations).

Pin: regress/contact-constrained-pendulum.dat (6,500 rows, sub-sampled into tests/golden/).  As with sitting-box.dat the file was
written by a Moby that already moved the body during the first step (row t = 0.001 shows y = -g dt^2 / 2); the current source
integrates positions with the pre-step velocity (TimeSteppingSimulator.cpp:155-164), so rows are compared one step later.  The
anchor point is not held exactly by either code (1.5 % off after 6.5 s in the file, 1.0 % here): the trajectories agree to 1.6e-3
over the first swing and to 2.4e-2 over all 6.5 s (two periods) -- a loose pin, stated as such."""
import os

import numpy as np
import pytest

import moby_sources
from moby_b200 import scenes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def hostsim():
    import hostsim_api
    hostsim_api.build()
    return hostsim_api


def _compare_with_golden(step_fn, get_pose):
    gold = np.loadtxt(os.path.join(GOLDEN, "regress_contact_constrained_pendulum.txt"))
    step, worst_first, worst = 0, 0.0, 0.0
    for row in gold:
        target = int(round(row[0] / 1e-3)) + 1                # one step later: see the module docstring
        step_fn(target - step)
        step = target
        err = np.abs(get_pose() - row[1:8]).max()
        worst = max(worst, err)
        if row[0] <= 2.0:
            worst_first = max(worst_first, err)
    return worst_first, worst


def test_oracle_matches_regress_contact_constrained_pendulum(oracle):
    sim = oracle.OracleSim(scenes.contact_constrained_pendulum(1))
    first, worst = _compare_with_golden(lambda n: sim.step(1e-3, n), lambda: sim.get_state()[0][0])
    assert first < 2e-3 and worst < 3e-2, (first, worst)
    c = sim.counters()
    assert c["lcp_failures"] == 0 and c["max_lcp_n"] == 48 and c["contacts"] == 6 * c["env_steps"] and c["stab_iterations"] > 0


def test_device_code_matches_oracle_on_the_pendulum(oracle, hostsim):
    """The solves are singular LCPs (the Lemke pivot paths of the tableau and the LU-per-pivot forms differ, tests/parity_util.py),
    but the net impulse is unique: the states agree to 1e-8 after 1,500 steps, fused and phased schedules bit for bit."""
    s = scenes.contact_constrained_pendulum(2)
    s.q[0, 0, 1] += 0.0                                           # two identical envs
    hf, hp = hostsim.HostSim(s), hostsim.HostSim(s)
    hf.step(1e-3, 1500)
    hp.step_phased(1e-3, 1500)
    assert np.array_equal(hf.q, hp.q) and np.array_equal(hf.v, hp.v)
    ob = oracle.OracleBatch(s)
    c = ob.run(1e-3, 1500, threads=2)
    q, v = ob.get_state_soa()
    assert np.abs(hf.q - q).max() < 1e-8 and np.abs(hf.v - v).max() < 1e-8
    assert hf.counters_dict()["lcp_failures"] == 0 and c["lcp_failures"] == 0
    assert hf.counters_dict()["lcp_solves"] == c["lcp_solves"] and hf.counters_dict()["contacts"] == c["contacts"]


@moby_sources.needed
def test_xml_pendulum_scene_loads_like_the_builder():
    from moby_b200 import xml_scene
    path = os.path.join(moby_sources.EXAMPLE, "contact-constrained-pendulum", "contact-constrained-pendulum.xml")
    s, info = xml_scene.load_xml(path, n_envs=1)
    b = scenes.contact_constrained_pendulum(1)
    assert info["bodies"] == {"l1": 0, "world": 1}
    for name in ("shape", "enabled", "mass", "dims", "inertia", "mu_coulomb", "epsilon", "NK", "q", "v"):
        assert np.allclose(getattr(s, name), getattr(b, name), atol=1e-12), name
    assert np.allclose(s.gravity, b.gravity) and s.stabilization_max_iterations == b.stabilization_max_iterations == 25
