"""The cost settings reach the kernels as data: every field of KinoSettings / PoseSettings lands in its slot of the
configuration tables that hb_kino_create receives (HB_KD_* doubles, HB_KI_* integers of include/hippopt_b200.h).

The tables are captured before they reach the library, so no GPU and no built library is needed.  The settings
are the distinct ones of tests_support: no two numbers are equal and none is 1, so a weight written to the wrong
slot, a dropped factor or two swapped weights show."""
import numpy as np
import pytest

from tests_support import KINO_MULTIPLIERS, POSE_MULTIPLIERS, distinct_cost_settings
from hippopt_b200._capi import H
from hippopt_b200.evaluator import KinoEvaluator, PoseEvaluator
from hippopt_b200.kino_layout import NJ, KinoSettings
from hippopt_b200.pose_layout import PoseSettings
from hippopt_b200.robot_model import ERGOCUB_JOINTS, RobotModel, synthetic_ergocub_urdf

# (foot frames, frame-cost frame, yaw points): the defaults, and geometries in which every body / point differs
GEOMETRIES = [(("l_sole", "r_sole"), "chest", (2, 3, 0)),
              (("r_sole", "l_sole"), "root_link", (0, 1, 2)),
              (("l_sole", "r_sole"), "l_sole", (3, 0, 1)),
              (("r_sole", "l_sole"), "l_forearm", (1, 3, 2))]


@pytest.fixture(scope="module")
def model():
    return RobotModel.from_urdf(synthetic_ergocub_urdf(), ERGOCUB_JOINTS, "root_link",
                                frames=["l_sole", "r_sole", "chest", "root_link", "l_forearm"])


@pytest.fixture
def captured(monkeypatch):
    """Evaluators built with this fixture keep (icfg, dcfg) instead of creating a library handle."""
    def keep(self, icfg, dcfg, lay):
        self.icfg, self.dcfg = icfg.copy(), dcfg.copy()

    monkeypatch.setattr(KinoEvaluator, "_create_handle", keep)
    monkeypatch.setattr(PoseEvaluator, "_create_handle", keep)


def kd_slot(name, n=1):
    o = H["HB_KD_" + name]
    return slice(o, o + n)


def check_geometry(ev, model, feet, frame):
    icfg, dcfg = ev.icfg, ev.dcfg
    assert icfg[H["HB_KI_FOOT_BODY_L"]] == model.frames[feet[0]][0]
    assert icfg[H["HB_KI_FOOT_BODY_R"]] == model.frames[feet[1]][0]
    assert icfg[H["HB_KI_CHEST_BODY"]] == model.frames[frame][0]
    for f in range(2):
        _, R, t = model.frames[feet[f]]
        assert np.array_equal(dcfg[kd_slot("FOOT_R0", 18)][9 * f:9 * f + 9], R.ravel())
        assert np.array_equal(dcfg[kd_slot("FOOT_T0", 6)][3 * f:3 * f + 3], t)
    assert np.array_equal(dcfg[kd_slot("CHEST_R0", 9)], model.frames[frame][1].ravel())


def test_geometries_are_distinct(model):
    """The frames of the geometries sit on five different bodies, the root among them, so a body taken from the
    wrong slot shows."""
    bodies = {fr: model.frames[fr][0] for fr in ("l_sole", "r_sole", "chest", "root_link", "l_forearm")}
    assert len(set(bodies.values())) == 5 and bodies["root_link"] == 0


@pytest.mark.parametrize("feet,frame,yaw", GEOMETRIES)
def test_kino_settings_land_in_their_slots(model, captured, feet, frame, yaw):
    d = distinct_cost_settings("kino")
    st = KinoSettings(horizon=3, final_state_constraint=True, foot_frames=feet, frame_quaternion_cost_frame=frame,
                      yaw_points=yaw, **d)
    ev = KinoEvaluator(model, st)
    dcfg = ev.dcfg
    slots = {"swing_foot_height_cost_multiplier": "W_SWING", "contact_velocity_control_cost_multiplier": "W_U",
             "contact_force_control_cost_multiplier": "W_FD", "contacts_centroid_cost_multiplier": "W_CENTROID",
             "desired_frame_quaternion_cost_multiplier": "W_FRAME", "base_quaternion_cost_multiplier": "W_BQ",
             "base_quaternion_velocity_cost_multiplier": "W_BQV", "joint_regularization_cost_multiplier": "W_JOINT",
             "force_regularization_cost_multiplier": "W_RATIO", "foot_yaw_regularization_cost_multiplier": "W_YAW"}
    assert set(slots) | {"com_linear_velocity_cost_multiplier"} == set(KINO_MULTIPLIERS)
    for name, slot in slots.items():
        assert dcfg[H["HB_KD_" + slot]] == d[name], name
    comvel = d["com_linear_velocity_cost_multiplier"] * np.asarray(d["com_linear_velocity_cost_weights"])
    assert np.array_equal(dcfg[kd_slot("W_COMVEL0", 3)], comvel)
    assert not np.array_equal(comvel, np.asarray(d["com_linear_velocity_cost_weights"]))  # the multiplier is not 1
    assert np.array_equal(dcfg[kd_slot("WJ0", NJ)], d["joint_regularization_cost_weights"])
    # every cost slot holds a different number: nothing was written twice
    w = dcfg[:H["HB_KD_WJ0"] + NJ]
    assert len(np.unique(w)) == len(w)
    icfg = ev.icfg
    assert tuple(icfg[H[k]] for k in ("HB_KI_YAW_BR", "HB_KI_YAW_TR", "HB_KI_YAW_TL")) == yaw
    check_geometry(ev, model, feet, frame)
    assert dcfg[H["HB_KD_TOTAL_MASS"]] == model.total_mass()


@pytest.mark.parametrize("feet,frame,yaw", GEOMETRIES)
def test_pose_settings_land_in_their_slots(model, captured, feet, frame, yaw):
    """The pose finder shares the weight slots of the kinodynamic table (csrc/pose_contact.cu header); the slots it
    has no cost for stay 0."""
    d = distinct_cost_settings("pose")
    ev = PoseEvaluator(model, PoseSettings(foot_frames=feet, frame_quaternion_cost_frame=frame, **d))
    dcfg = ev.dcfg
    slots = {"com_regularization_cost_multiplier": "W_CENTROID",
             "average_force_regularization_cost_multiplier": "W_RATIO",
             "point_position_regularization_cost_multiplier": "W_SWING",
             "force_regularization_cost_multiplier": "W_FD", "desired_frame_quaternion_cost_multiplier": "W_FRAME",
             "base_quaternion_cost_multiplier": "W_BQ", "joint_regularization_cost_multiplier": "W_JOINT"}
    assert set(slots) == set(POSE_MULTIPLIERS)
    for name, slot in slots.items():
        assert dcfg[H["HB_KD_" + slot]] == d[name], name
    assert np.array_equal(dcfg[kd_slot("WJ0", NJ)], d["joint_regularization_cost_weights"])
    for unused in ("W_U", "W_BQV", "W_YAW"):
        assert dcfg[H["HB_KD_" + unused]] == 0.0, unused
    assert not dcfg[kd_slot("W_COMVEL0", 3)].any()
    check_geometry(ev, model, feet, frame)


def test_default_settings_land_in_their_slots(model, captured):
    """The defaults go through the same path: W_COMVEL is the multiplier (1) times the weights (10, 0.1, 1)."""
    ev = KinoEvaluator(model, KinoSettings(horizon=2))
    assert np.array_equal(ev.dcfg[kd_slot("W_COMVEL0", 3)], [10.0, 0.1, 1.0])
    assert ev.dcfg[H["HB_KD_W_CENTROID"]] == 100.0 and ev.dcfg[H["HB_KD_W_YAW"]] == 2000.0
    pe = PoseEvaluator(model)
    assert pe.dcfg[H["HB_KD_W_SWING"]] == 100.0 and pe.dcfg[H["HB_KD_W_FD"]] == 0.2
