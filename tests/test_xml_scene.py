"""Moby XML scene loader (moby_b200/xml_scene.py): the reference's own example files load into the same batch
descriptors as the hand-written scene builders, and an inline scene steps on the oracle."""
import numpy as np
import pytest

import moby_sources
from moby_b200 import scenes, xml_scene

REF = moby_sources.EXAMPLE
needs_ref = moby_sources.needed

INLINE = """
<XML>
  <DRIVER step-size="0.001" />
  <MOBY>
    <Sphere id="s" radius="0.5" mass="2.0" />
    <Box id="b" xlen="1" ylen="0.5" zlen="2" density="3.0" />
    <Plane id="p" rpy="1.5707963267949 0 0" />
    <GravityForce id="g" accel="0 0 -9.81" />
    <RigidBody id="ball" position="0 0 2.0" linear-velocity="0.1 0 0" angular-velocity="0 0 1">
      <InertiaFromPrimitive primitive-id="s" /> <CollisionGeometry primitive-id="s" />
    </RigidBody>
    <RigidBody id="brick" position="3 0 1.0" quat="1 0 0 0">
      <InertiaFromPrimitive primitive-id="b" /> <CollisionGeometry primitive-id="b" />
    </RigidBody>
    <RigidBody id="ground" enabled="false" position="0 0 0"> <CollisionGeometry primitive-id="p" /> </RigidBody>
    <TimeSteppingSimulator min-step-size="1e-3" constraint-stabilization-max-iterations="0">
      <DynamicBody dynamic-body-id="ball" /> <DynamicBody dynamic-body-id="brick" /> <DynamicBody dynamic-body-id="ground" />
      <RecurrentForce recurrent-force-id="g" />
      <ContactParameters object1-id="ground" object2-id="ball" epsilon="0.5" mu-coulomb="0.2" friction-cone-edges="8" />
      <ContactParameters object1-id="brick" object2-id="ground" mu-coulomb="100" />
      <DisabledPair object1-id="ball" object2-id="brick" />
    </TimeSteppingSimulator>
  </MOBY>
</XML>
"""


def _same(a, b):
    for name in ("shape", "enabled", "mass", "dims", "inertia", "mu_coulomb", "mu_viscous", "epsilon", "compliance", "NK", "q", "v"):
        assert np.allclose(getattr(a, name), getattr(b, name), rtol=0, atol=1e-15), name
    assert tuple(a.gravity) == tuple(b.gravity) and a.min_step_size == b.min_step_size and a.contact_dist_thresh == b.contact_dist_thresh


@needs_ref
def test_reference_scenes_match_the_builders():
    s, info = xml_scene.load_xml(f"{REF}/simple-contact/simplest.xml", 3)
    _same(s, scenes.sitting_box(3, NK=8))
    assert info["bodies"] == {"box": 0, "ground": 1} and info["step_size"] == 0.1
    s, _ = xml_scene.load_xml(f"{REF}/bouncing-ball/bouncing-ball.xml", 2)
    _same(s, scenes.bouncing_ball(2))
    s, _ = xml_scene.load_xml(f"{REF}/stacks/sphere-stack.xml")
    _same(s, scenes.sphere_stack(1))
    s, _ = xml_scene.load_xml(f"{REF}/stacks/stack.xml")
    b = scenes.box_stack(1, 3, jitter=0.0, adjacent_only=False)
    _same(s, b)


@needs_ref
def test_unsupported_constructs_are_refused():
    with pytest.raises(ValueError):
        xml_scene.load_xml(f"{REF}/parts-feeder/feeder.xml")


def test_inline_scene(oracle):
    s, info = xml_scene.load_xml(INLINE, 2)
    assert info["bodies"] == {"ball": 0, "brick": 1, "ground": 2} and info["stabilization_max_iterations"] == 0
    assert s.gravity == (0.0, 0.0, -9.81) and s.min_step_size == 1e-3
    assert np.allclose(s.mass[:, 0], [2.0, 3.0, 1.0]) and np.allclose(s.inertia[0, :, 0], 0.4 * 2.0 * 0.25)
    assert np.allclose(s.inertia[1, :, 0], [3.0 * (0.25 + 4) / 12, 3.0 * (1 + 4) / 12, 3.0 * (1 + 0.25) / 12])
    nb = 3
    assert s.NK[0 * nb + 2, 0] == 8 and s.NK[1 * nb + 2, 0] == 4 and s.NK[0 * nb + 1, 0] == 0
    assert s.mu_coulomb[1 * nb + 2, 0] == 100.0 and s.epsilon[0 * nb + 2, 0] == 0.5
    assert np.allclose(s.v[0, :, 0], [0.1, 0, 0, 0, 0, 1])
    # the plane's primitive pose makes +z the normal: both bodies come to rest on it
    osim = oracle.OracleSim(s, 0)
    osim.step(1e-3, 4000)
    q, v = osim.get_state()
    assert abs(q[0, 2] - 0.5) < 1e-4 and abs(q[1, 2] - 1.0) < 1e-4
    assert osim.counters()["lcp_failures"] == 0
