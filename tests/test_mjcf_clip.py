"""G1-G3 of SURVEY Appendix G: the MJCF compiler and clip preprocessing against the ONLY numeric
pins the reference holds -- the derived fields of clips/transform_snips_groom.p (committed as
tests/golden/rodent_clip_golden.npz by tools/build_fixtures.py)."""
import numpy as np
import pytest

from conftest import pkg, reference_asset

mjcf = pkg("mjcf")
clipm = pkg("clip")

TRACKED = ["torso", "pelvis", "upper_leg_L", "lower_leg_L", "foot_L", "upper_leg_R", "lower_leg_R", "foot_R", "skull", "jaw",
           "scapula_L", "upper_arm_L", "lower_arm_L", "finger_L", "scapula_R", "upper_arm_R", "lower_arm_R", "finger_R"]


def test_rodent_dims(rodent):
    m, d = rodent["model"], rodent["dims"]
    # SURVEY Appendix A (parsed from assets/rodent.xml + envs/rodent.py:41-63)
    assert (m.nbody, m.njnt, m.nq, m.nv, m.nu, m.na, m.ngeom) == (66, 68, 74, 73, 30, 30, 101)
    assert (d["npair"], d["ncon"], d["nlimit"], d["nefc"]) == (32, 59, 67, 303)
    assert (d["nM"], d["nlevel"]) == (1119, 38)
    assert (d["solver"], d["iterations"], d["ls_iterations"], d["eulerdamp"]) == (1, 6, 6, 1)
    assert abs(m.timestep - 0.002) < 1e-12
    assert abs(float(m.arrays["body_mass"].sum()) - 0.186791) < 2e-6
    assert m.body_id("torso") == 1 and m.body_id("pelvis") == 8 and m.body_id("skull") == 54


def test_task_indices_reproduce_reference_quirks(rodent):
    idx, mb = rodent["idx"], pkg("model_blob")
    assert idx["end_eff_idx"] == [11, 15, 59, 64] and idx["app_idx"] == [11, 15, 59, 64, 54] and idx["com_idx"] == 1
    assert idx["body_idxs"] == [1, 8, 9, 10, 11, 13, 14, 15, 54, 55, 56, 57, 58, 60, 61, 62, 63, 65]
    assert len(idx["joint_idxs"]) == 33
    t = rodent["task_blob"]
    # Q5: filtered[:, app_idx] clamps to the 18-wide table; Q6: joint ids index nq-7 columns, id 67 clamps to 66
    assert mb.read_field(t, "VNL_T_APP_REF_IDX", np.int32).tolist() == [11, 15, 17, 17, 17]
    jc = mb.read_field(t, "VNL_T_JOINT_COL", np.int32)
    assert jc.tolist() == [min(j, 66) for j in idx["joint_idxs"]] and jc.max() == 66
    assert (rodent["obs_size"], rodent["traj_size"]) == (232, 795)  # notebooks/environments_explore.ipynb shapes


def test_fk_matches_clip_golden(rodent, golden):
    m = rodent["model"]
    ids = [m.body_id(n) for n in TRACKED]
    worst_p = worst_q = worst_c = 0.0
    for f in range(0, 250, 7):
        qpos = np.hstack([golden["position"][f], golden["quaternion"][f], golden["joints"][f]]).astype(np.float64)
        k = mjcf.kinematics(m, qpos)
        worst_p = max(worst_p, np.abs(k["xpos"][ids] - golden["body_positions"][f]).max())
        q, g = k["xquat"][ids], golden["body_quaternions"][f].astype(np.float64)
        s = np.sign((q * g).sum(1, keepdims=True))
        worst_q = max(worst_q, np.abs(q * s - g).max())
        com = mjcf.subtree_com(m, k["xipos"])[1]
        worst_c = max(worst_c, np.abs(com - golden["center_of_mass"][f]).max())
    assert worst_p < 1e-6 and worst_q < 1e-6 and worst_c < 1e-6, (worst_p, worst_q, worst_c)


def test_appendages_golden(rodent, golden):
    """walker.py:360-371 egocentric end effectors: (xpos[ee] - xpos[torso]) @ xmat[torso]."""
    m = rodent["model"]
    ee = [m.body_id(n) for n in ("lower_arm_R", "lower_arm_L", "foot_R", "foot_L", "skull")]
    for f in (0, 100, 249):
        qpos = np.hstack([golden["position"][f], golden["quaternion"][f], golden["joints"][f]]).astype(np.float64)
        k = mjcf.kinematics(m, qpos)
        app = (k["xpos"][ee] - k["xpos"][1]) @ k["xmat"][1]
        assert np.abs(app - golden["appendages"][f]).max() < 1e-6


def test_process_clip_matches_golden(rodent, golden):
    """process_clip restatement (preprocessing/mjx_preprocess.py:43-193): kinematic fields are the
    clip's own, velocities come from the finite-difference pipeline and are clipped to +-20."""
    c = rodent["clip"]
    assert c.body_positions.shape == (250, 66, 3)  # NEW clip format: all bodies (mjx_preprocess.py:126)
    ids = rodent["idx"]["body_idxs"]
    assert np.abs(c.body_positions[:, ids] - golden["body_positions"]).max() < 1e-6
    assert np.abs(c.position - golden["position"]).max() == 0
    assert np.abs(c.joints - golden["joints"]).max() == 0
    assert np.abs(c.velocity - golden["velocity"]).max() < 1e-6
    # angular velocity: fp32 arccos of a near-unit quaternion; the old (float64 MuJoCo) pipeline that wrote the
    # pickle resolves rotations below ~5e-4 rad/s that the fp32 process_clip rounds to zero (frame 219)
    dw = np.abs(c.angular_velocity - golden["angular_velocity"]).max(1)
    assert np.sort(dw)[-2] < 2e-5 and dw.max() < 5e-4
    assert np.abs(c.joints_velocity - golden["joints_velocity"]).max() < 1e-5
    assert np.abs(c.joints_velocity).max() <= 20.0
    assert np.abs(c.velocity[-1]).max() == 0  # padded last frame


def test_velocity_pipeline_from_qpos(golden):
    qpos = np.hstack([golden["position"], golden["quaternion"], golden["joints"]]).astype(np.float64)
    v = clipm.compute_velocity_from_kinematics(np.concatenate([qpos, qpos[-1:]]), 0.02)  # mjx_preprocess.py:88-90 pads
    assert v.shape == (250, 73)
    assert np.abs(v[:, :3] - golden["velocity"]).max() < 1e-6
    assert np.abs(np.clip(v[:, 6:], -20, 20) - golden["joints_velocity"]).max() < 1e-5


@pytest.mark.skipif(reference_asset("rodent.xml") is None, reason="no VNL_REFERENCE checkout of the original project")
def test_packaged_model_is_the_compiled_reference_asset(rodent):
    m2 = mjcf.load_rodent(reference_asset("rodent.xml"))
    m = rodent["model"]
    assert m2.body_names == m.body_names and m2.jnt_names == m.jnt_names
    for k, v in m.arrays.items():
        assert np.array_equal(np.asarray(m2.arrays[k]), np.asarray(v)), k


def test_humanoid_dims():
    """humanoid.xml as compiled by tools/build_fixtures.py into the packaged model."""
    m, _ = pkg("envs.humanoid").packaged_humanoid()
    d = pkg("model_blob").model_dims(m)
    assert (m.nbody, m.njnt, m.nq, m.nv, m.nu, m.na) == (17, 22, 28, 27, 21, 0)
    assert (d["ncon"], d["nlimit"], d["nefc"]) == (10, 21, 61)
    assert not m.eulerdamp and abs(m.timestep - 0.005) < 1e-12 and abs(m.impratio - 100.0) < 1e-9


def test_load_humanoid_recipe(tmp_path):
    """mjcf.load_humanoid on an MJCF file (envs/humanoid.py:40-54): compiled as written (no rescale), CG 6 x 6, eulerdamp
    disabled even where the file enables it."""
    import xml.etree.ElementTree as ET
    xml = ('<mujoco model="h"><option timestep="0.005" impratio="100"><flag eulerdamp="enable"/></option><worldbody>'
           '<geom name="floor" type="plane" size="5 5 0.1"/><body name="torso" pos="0 0 1.3"><freejoint name="root"/>'
           '<geom name="t" type="capsule" fromto="0 -.07 0 0 .07 0" size=".07"/><body name="arm" pos="0 0.2 0">'
           '<joint name="sh" type="hinge" axis="0 1 0" range="-60 60" damping="1"/>'
           '<geom name="a" type="capsule" fromto="0 0 0 0 0 -0.3" size="0.04"/></body></body></worldbody>'
           '<actuator><motor name="m" joint="sh" gear="40"/></actuator></mujoco>')
    path = tmp_path / "h.xml"
    path.write_text(xml)
    m = mjcf.load_humanoid(str(path))
    want = mjcf.compile_model(ET.fromstring(xml), name="humanoid", solver="cg", iterations=6, ls_iterations=6, eulerdamp=False)
    assert not m.eulerdamp and abs(m.timestep - 0.005) < 1e-12 and abs(m.impratio - 100.0) < 1e-9
    assert (m.solver, m.iterations, m.ls_iterations) == (want.solver, 6, 6) and (m.nq, m.nv, m.nu) == (8, 7, 1)
    assert m.body_names == want.body_names and m.arrays.keys() == want.arrays.keys()
    for k, v in want.arrays.items():
        assert np.array_equal(np.asarray(m.arrays[k]), np.asarray(v)), k
    assert np.allclose(m.arrays["jnt_range"][1], np.deg2rad([-60, 60]))  # degrees by default, as in humanoid.xml


def test_rescale_rule_only_touches_explicit_attributes():
    """dm_control rescale_subtree semantics (SURVEY Appendix D): default-class values are not scaled."""
    import xml.etree.ElementTree as ET
    root = ET.fromstring('<mujoco><default><joint pos="1 1 1"/></default><worldbody><body pos="1 2 3">'
                         '<joint name="a"/><geom size="2" pos="0 0 1"/><body pos="0 0 2"><joint name="b" pos="0 1 0"/></body>'
                         '</body></worldbody></mujoco>')
    mjcf.rescale_subtree(root, 0.5, 0.25)
    b = root.find("worldbody/body")
    assert b.get("pos").split() == ["0.5", "1", "1.5"] or np.allclose([float(x) for x in b.get("pos").split()], [0.5, 1, 1.5])
    assert np.allclose([float(x) for x in b.find("geom").get("size").split()], [0.5])
    assert b.find("joint").get("pos") is None
    assert np.allclose([float(x) for x in root.find("default/joint").get("pos").split()], [1, 1, 1])
    assert np.allclose([float(x) for x in b.find("body/joint").get("pos").split()], [0, 0.5, 0])
