"""Rimless wheel (example/rimless-wheel: wheel.xml, coldet-plugin.cpp, init.cpp; the other half of BASELINE configs[4]).

The wheel is a body whose collision geometry has no primitive; the reference's collision-detection plugin
(coldet-plugin.cpp:86-137,214-334) supplies its signed distance to the ground plane (lowest spoke tip), its contacts (one
per spoke tip below contact_dist_thresh) and an infinite "next" conservative-advancement step.  Here that plugin is the
shape SHAPE_WHEEL (dims = R, W, N_SPOKES).  mu = 100 sends every impact through the no-slip model.

Pin: regress/rimless-wheel.dat (6,275 rows, sub-sampled into tests/golden/regress_rimless_wheel.txt).  The file was written
by a configuration the tree no longer holds -- with today's wheel.xml (alpha = 0.1, Iyy = 1) and init.cpp the wheel does
not follow it.  The recorded motion itself identifies the configuration: the centre stays at distance R = 1 (1e-6) from
the fixed point (0.5, 0, 0) -- spoke tip 5 pinned by the no-slip contact -- and the angular acceleration over the swing is
that of a pendulum with g = (0.0500, 0, -0.9987) (wheel.xml:15, its own "alpha = 0.05" alternative) and
|g| / I_tip = 0.33335, i.e. Iyy = 2 with m = R = 1.  The initial spin is not recorded either; one number (omega_0) is fitted.
With those three reconstructed values the restated path reproduces all 6,275 rows of all 7 coordinates to 1.1e-5 over 6.27 s
of no-slip contact solves and constraint stabilization: "pinned with a reconstructed configuration", and said so here.
"""
import os

import numpy as np
import pytest

import moby_sources
from moby_b200 import scenes

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
G_ALPHA_005 = (0.049979, 0.0, -0.99875)          # wheel.xml:15
OMEGA_0 = 0.2892051330771366                     # fitted once against the golden rows (see the module docstring)
S60, C60 = 0.866025403784439, 0.5


def golden_scene(n_envs=1):
    s = scenes.rimless_wheel(n_envs, theta_dot=0.0, alpha_gravity=G_ALPHA_005, inertia=(2.0, 2.0, 2.0))
    s.v[1, 0, :], s.v[1, 2, :], s.v[1, 4, :] = OMEGA_0 * S60, OMEGA_0 * C60, OMEGA_0     # rolling about spoke tip 5
    return s


@pytest.fixture(scope="module")
def hostsim():
    import hostsim_api
    hostsim_api.build()
    return hostsim_api


def test_wheel_plane_distance_and_contacts(oracle):
    """coldet-plugin.cpp:86-137: distance = lowest tip height; :222-310: one contact per tip below the threshold, at the
    midpoint of tip and projection, normal = plane +Y, signed violation = the tip height."""
    s = scenes.rimless_wheel(1, theta_dot=0.0)
    s.q[1, 2, :] = 0.9                         # tips 4 and 5 are 0.9 - sin 60 = 0.03397 above the ground: no contact
    o = oracle.OracleSim(s)
    o.step(1e-9)
    assert o.counters()["contacts"] == 0
    s.q[1, 2, :] = S60 - 1e-4                  # both tips 1e-4 deep
    o = oracle.OracleSim(s)
    o.step(1e-9)
    con = o.last_contacts()
    assert con["count"] == 2
    for i, tip_x in enumerate((-0.5, 0.5)):    # spoke 4 (240 deg) then spoke 5 (300 deg)
        assert np.allclose(con["normal"][i], (0, 0, 1), atol=1e-9)
        assert np.allclose(con["point"][i], (tip_x, 0.0, -0.5e-4), atol=1e-9)
        assert abs(con["dist"][i] + 1e-4) < 1e-9


def test_oracle_matches_regress_rimless_wheel(oracle):
    gold = np.loadtxt(os.path.join(GOLDEN, "regress_rimless_wheel.txt"))
    sim = oracle.OracleSim(golden_scene())
    step, worst = 0, 0.0
    for row in gold:
        target = int(round(row[0] / 1e-3))
        sim.step(1e-3, target - step)
        step = target
        q, _ = sim.get_state()
        worst = max(worst, np.abs(q[1] - row[1:8]).max())
    assert worst < 2e-5, worst
    c = sim.counters()
    assert c["lcp_failures"] == 0 and c["lemke_calls"] == 0 and c["stab_line_search_failures"] == 0
    assert c["lcp_solves"] > 5000            # a no-slip impact solve on most steps: the tip contact is re-established every step


@pytest.mark.parametrize("stab", [0, -1])
def test_device_code_matches_oracle_on_wheels(oracle, hostsim, stab):
    """A batch of wheels with random spins: the kernels' device code (host build), fused and phased, against the oracle,
    across several spoke-to-spoke impacts (0.6 s at up to 4.5 rad/s is more than one spoke period)."""
    ne = 12
    s = scenes.rimless_wheel(ne, theta_dot=3.0, seed=5, stabilization=stab)
    hs, hp = hostsim.HostSim(s), hostsim.HostSim(s)
    hs.step(1e-3, 600)
    hp.step_phased(1e-3, 600)
    assert np.array_equal(hs.q, hp.q) and np.array_equal(hs.v, hp.v)
    ob = oracle.OracleBatch(s)
    c = ob.run(1e-3, 600, threads=4)
    q, v = ob.get_state_soa()
    assert np.abs(hs.q - q).max() < 1e-12 and np.abs(hs.v - v).max() < 1e-11
    ch = hs.counters_dict()
    for k in ("mini_steps", "lcp_solves", "lcp_fast_calls", "lemke_calls", "lcp_failures", "contacts", "stab_iterations"):
        assert ch[k] == c[k], (k, ch[k], c[k])
    assert c["lcp_failures"] == 0
    assert (q[1, 0, :] > 0.5).all()          # every wheel rolled past its first spoke


@moby_sources.needed
def test_xml_wheel_scene_loads_like_the_builder():
    from moby_b200 import xml_scene
    path = os.path.join(moby_sources.EXAMPLE, "rimless-wheel", "wheel.xml")
    s, info = xml_scene.load_xml(path, n_envs=1)
    assert info["bodies"] == {"GROUND": 0, "WHEEL": 1}
    b = scenes.rimless_wheel(1, theta_dot=0.0)
    b.q[1, 2, :] = 1.0                        # wheel.xml:42 (the initializer plugin moves it to sin 60 deg)
    for name in ("shape", "enabled", "mass", "dims", "inertia", "mu_coulomb", "epsilon", "NK", "q", "v"):
        assert np.allclose(getattr(s, name), getattr(b, name), atol=1e-12), name
    assert np.allclose(s.gravity, b.gravity) and s.stabilization_max_iterations == b.stabilization_max_iterations
