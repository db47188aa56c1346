"""MJCF reader + canonical tree (host logic; no GPU)."""
import os

import numpy as np
import pytest

from conftest import ASSET, GOLDEN, NEUTRAL, tree_fk
from mujoco_panda_pnp_b200 import KinematicData, KinematicModel, KinematicTree
from mujoco_panda_pnp_b200.mjcf import JNT_FREE, JNT_HINGE, JNT_SLIDE
from oracle import ik_oracle, mj_oracle

HOME_WPT = np.array([1.23843967, 0.0, 0.49740014])  # real MuJoCo, scripts/execute_pnp.py:38


def test_fk_neutral_matches_real_mujoco_value():
    tree = KinematicTree.from_mjcf()
    assert np.abs(tree_fk(tree, NEUTRAL) - HOME_WPT).max() < 1e-8
    assert np.allclose(tree_fk(tree, np.zeros(7)), [0.688, 0.0, 1.121], atol=1e-12)


def test_model_layout_matches_reference_scene(kin_model):
    m = kin_model
    assert (m.nq, m.nv, m.njnt) == (37, 33, 13)  # SURVEY App. A
    assert m.joint_names[:9] == [f"joint{i}" for i in range(1, 8)] + ["finger_joint1", "finger_joint2"]
    assert list(m.jnt_type[:7]) == [JNT_HINGE] * 7 and list(m.jnt_type[7:9]) == [JNT_SLIDE] * 2
    assert list(m.jnt_type[9:]) == [JNT_FREE] * 4
    assert list(m.jnt_qposadr) == [0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 16, 23, 30]
    np.testing.assert_allclose(m.jnt_range[:7, 0], [-2.8973, -1.7628, -2.8973, -3.0718, -2.8973, -0.0175, -2.8973])
    np.testing.assert_allclose(m.jnt_range[:7, 1], [2.8973, 1.7628, 2.8973, -0.0698, 2.8973, 3.7525, 2.8973])
    np.testing.assert_allclose(m.jnt_range[7:9], [[0, 0.04]] * 2)
    np.testing.assert_allclose(m.jnt_axis[7], [0, 1, 0])
    # free-joint qpos0 = body pos + quat (cube1 at 1.4 0 0.73)
    np.testing.assert_allclose(m.qpos0[9:16], [1.4, 0, 0.73, 1, 0, 0, 0])
    assert m.site("ee_center_site").id == 0
    np.testing.assert_allclose(m.site_pos[m.site("target_cube1").id], [1.0, -0.1, 0.3])
    assert m.opt.timestep == 0.002
    with pytest.raises(KeyError):
        m.site("nope")


def test_packaged_asset_equals_reference_mjcf():
    """tests/golden/reference_scene_golden.npz holds what the loader reads from the reference's
    assets/shelf_pnp.xml (+ panda_mocap.xml): the model fields, the names and the canonical tree.  They were
    recorded from the packaged asset, which had been checked field for field equal to the reference's MJCF and
    whose bodies, joints and sites have not changed since."""
    ours = KinematicModel.from_xml_path(ASSET)
    ref = np.load(os.path.join(GOLDEN, "reference_scene_golden.npz"))
    for f in ("body_parentid", "body_pos", "body_quat", "body_jntadr", "body_jntnum", "jnt_type", "jnt_axis",
              "jnt_pos", "jnt_qposadr", "jnt_dofadr", "jnt_range", "qpos0", "site_bodyid", "site_pos", "site_quat"):
        np.testing.assert_array_equal(getattr(ours, f), ref[f], err_msg=f)
    assert ours.body_names == ref["body_names"].tolist() and ours.joint_names == ref["joint_names"].tolist()
    assert ours.site_names == ref["site_names"].tolist()
    assert bytes(KinematicTree.from_mjmodel(ours).to_struct()) == ref["tree_struct"].tobytes()


def test_from_mjmodel_accepts_foreign_model_objects(oracle_model):
    """The loader only relies on MjModel field names: the oracle's independent MJCF compile
    (a different class) must give the identical canonical tree."""
    t1 = KinematicTree.from_mjmodel(oracle_model)
    t2 = KinematicTree.from_mjcf()
    assert bytes(t1.to_struct()) == bytes(t2.to_struct())
    assert t1.body_chain == [oracle_model.body(n).id for n in
                             ["link0", "link1", "link2", "link3", "link4", "link5", "link6", "link7", "hand",
                              "ee_center_body"]]


def test_canonical_form_is_z_hinges():
    t = KinematicTree.from_mjcf()
    assert t.link_pos.shape == (7, 3) and t.link_rot.shape == (7, 3, 3)
    for r in t.link_rot:
        np.testing.assert_allclose(r @ r.T, np.eye(3), atol=1e-15)
    np.testing.assert_allclose(t.link_pos[0], [0.6, 0, 0.633])  # link0 folded into joint1's frame
    np.testing.assert_allclose(t.ee_pos, [0, 0, 0.212])  # hand + ee_center_body folded
    s = t.snapped()
    assert set(np.unique(np.abs(s.link_rot))) <= {0.0, 1.0}
    assert np.abs(s.link_rot - t.link_rot).max() < 1e-15


_GENERAL_MJCF = """
<mujoco>
  <compiler angle="degree"/>
  <default><joint range="-170 170"/></default>
  <worldbody>
    <body name="b0" pos="0.1 0.2 0.3" euler="10 20 30">
      <body name="b1" pos="0 0 0.2" quat="0.9 0.1 -0.2 0.3">
        <joint name="j1" axis="1 1 0" pos="0.01 0.02 0.03"/>
        <body name="b2" pos="0.1 0 0.1" axisangle="0 1 0 35">
          <joint name="j2" axis="0 1 0" pos="0 0.05 0" ref="15"/>
          <body name="b3" pos="0 0.2 0">
            <joint name="j3" axis="0 0 -1"/>
            <body name="b4" pos="0.05 0 0.1" quat="1 0 1 0">
              <joint name="j4" axis="1 0 0" range="-90 45"/>
              <body name="b5" pos="0 0 0.15">
                <joint name="j5" axis="0.3 -0.4 0.5" pos="0.02 0 0"/>
                <body name="b6" pos="0.02 0.03 0.1">
                  <joint name="j6" axis="0 1 0"/>
                  <body name="b7" pos="0 0 0.08" quat="0.7 0 0.7 0.1">
                    <joint name="j7" axis="0 0 1" pos="0 0.01 0"/>
                    <body name="tool" pos="0.01 0.02 0.1" quat="1 0.2 0 0">
                      <site name="ee_center_site" pos="0.01 0 0.05" quat="0.8 0 0.6 0"/>
                    </body>
                  </body>
                </body>
              </body>
            </body>
          </body>
        </body>
      </body>
    </body>
  </worldbody>
</mujoco>
"""


def test_general_tree_folding_matches_mujoco_semantics(tmp_path):
    """Arbitrary hinge axes, non-zero jnt_pos, ref angles, euler/axisangle frames, degrees:
    the canonical z-hinge chain must reproduce mj_kinematics (oracle) exactly."""
    p = tmp_path / "general.xml"
    p.write_text(_GENERAL_MJCF)
    model = KinematicModel.from_xml_path(str(p))
    tree = KinematicTree.from_mjmodel(model)
    np.testing.assert_allclose(tree.qref[1], np.deg2rad(15))
    np.testing.assert_allclose(tree.lower[3], np.deg2rad(-90))
    # oracle kinematics run on the product's parsed model (oracle reader is quat-only)
    data = mj_oracle.MjData(model)
    data.xanchor = np.zeros((model.njnt, 3))
    rng = np.random.default_rng(5)
    for _ in range(20):
        q = rng.uniform(-2.5, 2.5, 7)
        want = ik_oracle.fk_site(model, data, q)[0]
        np.testing.assert_allclose(tree_fk(tree, q), want, atol=1e-13)


def test_kinematic_data_mimics_mjdata(kin_model):
    d = KinematicData(kin_model)
    assert d.qpos.shape == (37,) and d.qvel.shape == (33,)
    assert d.site_xpos.shape == (7, 3)


def test_loader_rejects_unsupported_chains(tmp_path):
    bad = tmp_path / "bad.xml"
    bad.write_text("<mujoco><worldbody><body><joint type='slide'/><site name='ee_center_site'/></body></worldbody></mujoco>")
    with pytest.raises(ValueError):
        KinematicTree.from_mjcf(str(bad))
