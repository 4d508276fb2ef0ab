"""SDF subset reader (moby_b200/sdf_scene.py) against example/ur10/model.sdf: the kinematic / inertial tables scenes.ur10 is
built from were transcribed from that file by hand; parsed, they must come out the same."""
import os

import numpy as np
import pytest

import moby_sources
from moby_b200 import scenes, sdf_scene

SDF = os.path.join(moby_sources.EXAMPLE, "ur10", "model.sdf")


@moby_sources.needed
def test_ur10_sdf_matches_the_transcribed_tables():
    name, links, joints = sdf_scene.load_sdf_model(SDF)
    assert name == "ur10_schunk_hybrid" and len(links) == len(scenes._UR10_LINKS) == 10
    for got, want in zip(links, scenes._UR10_LINKS):
        assert got[0] == want[0]
        assert np.array_equal(np.array(got[1]), np.array(want[1], float)) and np.array_equal(np.array(got[2]), np.array(want[2], float))
        assert got[3] == want[3] and np.array_equal(np.array(got[4]), np.array(want[4]))
    assert joints[0]["parent"] == "world" and joints[0]["upper"] == 1e-5           # world_joint: a weld by +-1e-5 limits
    for k in range(1, 10):
        parent, jtype, axis = scenes._UR10_JOINTS[k]
        assert joints[k]["parent"] == parent and joints[k]["type"] == jtype
        assert np.allclose(joints[k]["axis"], axis, atol=2e-5), (k, joints[k]["axis"], axis)     # rpy values carry 6 digits
    assert [j["name"] for j in joints[1:7]] == ["shoulder_pan_joint", "shoulder_lift_joint", "elbow_joint", "wrist_1_joint", "wrist_2_joint", "wrist_3_joint"]
    assert joints[7]["upper"] == 1e-5 and joints[8]["type"] == scenes.JOINT_PRISMATIC    # hand weld and the finger slides, limits recorded


def test_sdf_reader_refuses_what_it_cannot_represent(tmp_path):
    p = tmp_path / "m.sdf"
    p.write_text("<sdf version='1.5'><model name='m'><link name='a'><inertial><mass>1</mass><inertia><ixx>1</ixx><ixy>0.1</ixy><ixz>0</ixz>"
                 "<iyy>1</iyy><iyz>0</iyz><izz>1</izz></inertia></inertial></link></model></sdf>")
    with pytest.raises(ValueError, match="off-diagonal"):
        sdf_scene.load_sdf_model(str(p))
    p.write_text("<sdf version='1.5'><model name='m'><link name='a'><inertial><mass>1</mass><inertia><ixx>1</ixx><ixy>0</ixy><ixz>0</ixz>"
                 "<iyy>1</iyy><iyz>0</iyz><izz>1</izz></inertia></inertial></link><link name='b'><inertial><mass>1</mass><inertia><ixx>1</ixx>"
                 "<ixy>0</ixy><ixz>0</ixz><iyy>1</iyy><iyz>0</iyz><izz>1</izz></inertia></inertial></link>"
                 "<joint name='j' type='ball'><parent>a</parent><child>b</child><axis><xyz>0 0 1</xyz></axis></joint></model></sdf>")
    with pytest.raises(ValueError, match="ball"):
        sdf_scene.load_sdf_model(str(p))
