"""The C++ host facade (include/b200moby.hpp, Moby's class names over the C ABI): builds with plain g++ against
libb200moby.so; without a GPU the program fails loudly (no CPU fallback); on the GPU it reproduces the oracle."""
import os
import subprocess

import numpy as np
import pytest

import moby_sources

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CPP = os.path.join(ROOT, "tests", "cpp")


@pytest.fixture(scope="module")
def sitting_box():
    import __graft_entry__ as g
    from moby_b200 import capi
    if not os.path.exists(capi.LIB_PATH):
        g.build()
    subprocess.check_call(["make", "-s", "-C", CPP])
    return os.path.join(CPP, "sitting_box")


def test_facade_builds_and_refuses_without_gpu(sitting_box):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([sitting_box, "10", "5"], capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_facade_sitting_box_matches_oracle(sitting_box, oracle):
    from moby_b200 import scenes
    r = subprocess.run([sitting_box, "400", "100", "3"], capture_output=True, text=True, check=True)
    rows = [l.split() for l in r.stdout.splitlines() if l and not l.startswith("#")]
    osim = oracle.OracleSim(scenes.sitting_box(1, NK=8, y0=0.50001))
    k = 0
    for step in range(1, 401):
        osim.step(1e-3)
        if step % 100 == 0:
            qo, _ = osim.get_state()
            for _ in range(2):                       # env 0 and env n-1 are printed; both are the same scene
                row = rows[k]; k += 1
                assert abs(float(row[0]) - step * 1e-3) < 1e-12
                assert np.array_equal(np.array([float(x) for x in row[2:9]]), qo[0])
    meta = {l.split()[1]: l.split()[2:] for l in r.stdout.splitlines() if l.startswith("#")}
    assert meta["env_steps"][0] == "1200" and meta["env_steps"][-1] == "400"          # 3 envs x 400 steps; 400 callbacks
    zl = [float(x) for x in meta["lcp_lemke"][1:]]
    zf = [float(x) for x in meta["lcp_fast"][1:]]
    assert meta["lcp_lemke"][0] == "1" and np.allclose(zl, [4 / 3, 7 / 3], atol=1e-14)
    assert meta["lcp_fast"][0] == "1" and np.allclose(zf, [4 / 3, 7 / 3], atol=1e-14)


# ---- Moby::XMLReader::read of the facade (include/b200moby_xml.hpp) against the Python loader ----
REF = moby_sources.EXAMPLE


def _dump(sitting_box, path):
    exe = os.path.join(CPP, "xml_dump")
    r = subprocess.run([exe, path], capture_output=True, text=True)
    return r.returncode, r.stdout, r.stderr


def _check_against_python_loader(sitting_box, path):
    from moby_b200 import xml_scene
    rc, out, err = _dump(sitting_box, path)
    assert rc == 0, err
    s, info = xml_scene.load_xml(path, 1)
    nb = s.n_bodies
    lines = out.splitlines()
    head = lines[0].split()
    assert float(head[3]) == s.min_step_size and float(head[5]) == s.contact_dist_thresh
    bodies = [l.split() for l in lines if l.startswith("body ")]
    assert [b[2] for b in bodies] == sorted(info["bodies"], key=info["bodies"].get)
    for i, b in enumerate(bodies):
        f = lambda k, n: np.array([float(x) for x in b[k:k + n]])  # noqa: E731
        assert int(b[4]) == s.enabled[i, 0] and int(b[6]) == s.shape[i, 0]
        assert np.array_equal(f(8, 3), s.dims[i, :, 0])
        assert np.allclose(f(18, 7), s.q[i, :, 0], rtol=0, atol=1e-15) and np.array_equal(f(26, 6), s.v[i, :, 0])
        assert np.array_equal(f(33, 3), np.array(s.gravity))
        if s.enabled[i, 0]:
            assert np.allclose(float(b[12]), s.mass[i, 0], rtol=1e-15) and np.allclose(f(14, 3), s.inertia[i, :, 0], rtol=1e-15)
    seen = set()
    for l in lines:
        if not l.startswith("contact "):
            continue
        t = l.split()
        a, b = int(t[1]), int(t[2])
        o = a * nb + b
        seen.add(o)
        assert float(t[4]) == s.epsilon[o, 0] and float(t[6]) == s.mu_coulomb[o, 0] and float(t[8]) == s.mu_viscous[o, 0]
        assert float(t[10]) == s.compliance[o, 0] and int(t[12]) == s.NK[o, 0]
    for a in range(nb):                                   # pairs the file does not mention keep the defaults in both loaders
        for b in range(a + 1, nb):
            if a * nb + b not in seen:
                assert s.NK[a * nb + b, 0] == 4 and s.mu_coulomb[a * nb + b, 0] == 0.0 and s.epsilon[a * nb + b, 0] == 0.0


@moby_sources.needed
@pytest.mark.parametrize("rel", ["simple-contact/simplest.xml", "bouncing-ball/bouncing-ball.xml", "stacks/sphere-stack.xml", "stacks/stack.xml",
                                 "rimless-wheel/wheel.xml", "contact-constrained-pendulum/contact-constrained-pendulum.xml"])
def test_cpp_xml_reader_loads_reference_scenes(sitting_box, rel):
    _check_against_python_loader(sitting_box, os.path.join(REF, rel))


def test_cpp_xml_reader_inline_scene_and_errors(sitting_box, tmp_path):
    from test_xml_scene import INLINE
    good = tmp_path / "scene.xml"
    good.write_text(INLINE.replace('<DisabledPair object1-id="ball" object2-id="brick" />', ""))
    _check_against_python_loader(sitting_box, str(good))
    bad = tmp_path / "joint.xml"
    bad.write_text(INLINE.replace("<GravityForce", '<RevoluteJoint id="j" /> <GravityForce'))
    rc, out, err = _dump(sitting_box, str(bad))
    assert rc == 1 and "RevoluteJoint" in err
    broken = tmp_path / "broken.xml"
    broken.write_text("<XML><MOBY><Box id='b' xlen='1'></MOBY></XML>")
    rc, out, err = _dump(sitting_box, str(broken))
    assert rc == 1 and "XML parse error" in err


# ---- articulated bodies, controller callback, constraint callback, extern "C" init plugin (SURVEY.md 8b; VERDICT r01 #9) ----
def test_pendulum_and_plugin_driver_build_and_refuse_without_gpu(sitting_box):
    """example/sims-in-code/pendulum.cpp and a controller plugin shaped like example/ur10/controller.cpp compile against the
    facade; without a GPU both programs stop at b200moby_create."""
    import torch
    for exe in ("pendulum", "plugin_driver", "libctrl_plugin.so"):
        assert os.path.exists(os.path.join(CPP, exe)), exe
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = subprocess.run([os.path.join(CPP, "pendulum"), "10", "5"], capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr
    r = subprocess.run([os.path.join(CPP, "plugin_driver"), os.path.join(CPP, "libctrl_plugin.so"), "10", "5"], capture_output=True, text=True)
    assert r.returncode == 3 and "no CPU fallback" in r.stderr


def _arm2_scene(n_envs=1, controller=True):
    """The scene tests/cpp/plugin_driver.cpp builds through the facade, built with the Python mirror."""
    from moby_b200 import scenes
    s = scenes.SceneBatch(n_envs, 5)
    s.gravity = (0.0, 0.0, -9.81)
    m, dx, dy, dz = 1.0, 0.5, 0.05, 0.05
    for b, cx in enumerate((0.0, 0.25, 0.75)):
        s.mass[b, :] = m
        s.inertia[b, 0, :], s.inertia[b, 1, :], s.inertia[b, 2, :] = m * (dy * dy + dz * dz) / 12, m * (dx * dx + dz * dz) / 12, m * (dx * dx + dy * dy) / 12
        s.q[b, 0, :], s.q[b, 2, :] = cx, 1.0
    rc = scenes.ArticulatedBody(s, 0, 3, fdyn=scenes.FDYN_CRB)
    rc.set_joint(1, 0, scenes.JOINT_REVOLUTE, (0, 1, 0), (0.0, 0, 0), (-0.25, 0, 0))
    rc.set_joint(2, 1, scenes.JOINT_REVOLUTE, (0, 1, 0), (0.25, 0, 0), (-0.25, 0, 0))
    if controller:
        rc.set_controller(kp=[30.0, 10.0], kv=[6.0, 2.0], amp=[0.5, 0.3], freq=[1.0, 2.0])
    rc.jqd[0, :], rc.jqd[1, :] = 0.5, 0.3
    s.set_sphere(3, 0.1, mass=1.0)
    s.q[3, 0, :], s.q[3, 2, :] = 2.0, 0.1
    h = np.sqrt(0.5)
    s.set_plane(4, quat=(h, 0, 0, h))
    for i in range(5):
        for j in range(i + 1, 5):
            s.set_contact(i, j)
    return s


@pytest.mark.gpu
def test_plugin_controller_matches_builtin_pd_law(sitting_box):
    """The plugin's controller (host callback every step -> b200moby_set_joint_forces) against the same PD law evaluated on
    the device (rc.set_controller): joint trajectories agree to 1e-9; the constraint callback saw the ball's contact every step."""
    from moby_b200 import TimeSteppingSimulator
    r = subprocess.run([os.path.join(CPP, "plugin_driver"), os.path.join(CPP, "libctrl_plugin.so"), "300", "100"], capture_output=True, text=True, check=True)
    rows = [[float(x) for x in l.split()] for l in r.stdout.splitlines() if l and not l.startswith("#")]
    meta = [l.split() for l in r.stdout.splitlines() if l.startswith("#")][0]
    assert int(meta[2]) == 300 and int(meta[4]) >= 1
    sim = TimeSteppingSimulator(_arm2_scene())
    for k, row in enumerate(rows):
        sim.step(1e-3, 100)
        jq, jqd = sim.get_joint_state()
        q, _ = sim.get_state()
        got = np.array([jq[0, 0], jq[1, 0], jqd[0, 0], jqd[1, 0], q[3, 2, 0]])
        assert abs(row[0] - (k + 1) * 0.1) < 1e-12
        assert np.allclose(got, row[1:6], rtol=0, atol=1e-9), (got, row[1:6])
    assert abs(rows[-1][1]) > 1e-3            # the arm did move


@pytest.mark.gpu
def test_facade_pendulum_matches_python_mirror(sitting_box):
    from moby_b200 import TimeSteppingSimulator, scenes
    r = subprocess.run([os.path.join(CPP, "pendulum"), "400", "200", "2"], capture_output=True, text=True, check=True)
    rows = [[float(x) for x in l.split()] for l in r.stdout.splitlines() if l]
    s = scenes.SceneBatch(1, 2)
    s.gravity = (0.0, 0.0, -9.8)
    s.mass[:, :] = 1.0
    s.inertia[0, :, :] = 1.0 * (0.01 + 0.01) / 12
    s.inertia[1, 0, :] = s.inertia[1, 2, :] = (3 * 0.025 ** 2 + 1.0) / 12.0
    s.inertia[1, 1, :] = 0.5 * 0.025 ** 2
    s.q[1, 1, :] = -0.5
    rc = scenes.ArticulatedBody(s, 0, 2, fdyn=scenes.FDYN_CRB)
    rc.set_joint(1, 0, scenes.JOINT_REVOLUTE, (1, 0, 0), (0, 0, 0), (0, 0.5, 0))
    s.stabilization_max_iterations = -1
    sim = TimeSteppingSimulator(s)
    for row in rows:
        sim.step(1e-3, 200)
        q, _ = sim.get_state()
        jq, jqd = sim.get_joint_state()
        assert np.allclose(q[1, :, 0], row[1:8], rtol=0, atol=1e-12) and abs(jq[0, 0] - row[8]) < 1e-12 and abs(jqd[0, 0] - row[9]) < 1e-12
