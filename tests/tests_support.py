"""Shared helpers of the test suite."""
import dataclasses
import glob
import os

import numpy as np

GOLD = os.path.join(os.path.dirname(__file__), "golden")

# the cost multipliers of each planner: every one scales exactly one family of cost expressions
KINO_MULTIPLIERS = (
    "contacts_centroid_cost_multiplier", "com_linear_velocity_cost_multiplier",
    "desired_frame_quaternion_cost_multiplier", "base_quaternion_cost_multiplier",
    "base_quaternion_velocity_cost_multiplier", "joint_regularization_cost_multiplier",
    "force_regularization_cost_multiplier", "foot_yaw_regularization_cost_multiplier",
    "swing_foot_height_cost_multiplier", "contact_velocity_control_cost_multiplier",
    "contact_force_control_cost_multiplier")
POSE_MULTIPLIERS = (
    "base_quaternion_cost_multiplier", "desired_frame_quaternion_cost_multiplier",
    "joint_regularization_cost_multiplier", "force_regularization_cost_multiplier",
    "com_regularization_cost_multiplier", "average_force_regularization_cost_multiplier",
    "point_position_regularization_cost_multiplier")


def distinct_cost_settings(kind: str) -> dict:
    """Cost settings in which no two numbers are equal and none is 1, so that a weight read from the wrong slot, a
    dropped factor or two swapped weights change the result.  The multipliers are spread log-uniformly over
    1e-3 ... 1e3 in a shuffled order; the 23 joint weights (and, for the kinodynamic problem, the 3 CoM-velocity
    weights) are distinct values in 0.2 ... 5, away from every multiplier."""
    rng = np.random.default_rng(11 if kind == "kino" else 12)
    names = KINO_MULTIPLIERS if kind == "kino" else POSE_MULTIPLIERS
    expo = np.linspace(-3.0, 3.0, len(names)) + 0.0731  # +0.0731: no multiplier is 1 (exponent 0)
    out = {n: float(10.0 ** e) for n, e in zip(names, rng.permutation(expo))}
    w = 10.0 ** rng.permutation(np.linspace(np.log10(0.2), np.log10(5.0), 26) + 0.0173)
    out["joint_regularization_cost_weights"] = w[:23]
    if kind == "kino":
        out["com_linear_velocity_cost_weights"] = tuple(float(v) for v in w[23:])
    vals = [v for v in out.values() if np.isscalar(v)] + list(w if kind == "kino" else w[:23])
    assert len(set(vals)) == len(vals) and 1.0 not in vals
    return out


def only_term(kind: str, name: str | None) -> dict:
    """The distinct settings with every multiplier but ``name`` set to 0 (all of them for name=None)."""
    s = distinct_cost_settings(kind)
    for n in (KINO_MULTIPLIERS if kind == "kino" else POSE_MULTIPLIERS):
        if n != name:
            s[n] = 0.0
    return s


def oracle_settings(cls, settings, **extra):
    """An instance of the oracle's settings dataclass ``cls`` that copies every field it shares with an evaluator
    settings object (KinoSettings / PoseSettings); the kinodynamic yaw points are spelled out as the oracle names
    them, and the terrain (a name on one side, an expression on the other) comes in ``extra``."""
    names = {f.name for f in dataclasses.fields(cls)} - {"terrain"}
    kw = {f.name: getattr(settings, f.name) for f in dataclasses.fields(settings) if f.name in names}
    if hasattr(settings, "yaw_points"):
        kw["yaw_bottom_right"], kw["yaw_top_right"], kw["yaw_top_left"] = settings.yaw_points
    return cls(**kw, **extra)


def golden_files(kind: str, extra_dirs=()):
    """Golden fixtures of one problem kind ("kino", "toy"): the committed oracle-generated files AND, when present,
    the CasADi dumps `casadi_<kind>_*.npz` written by tools/dump_casadi_golden.py in the reference environment --
    both are compared with the CUDA path / the oracle by the same tests."""
    out = []
    for d in (GOLD, *extra_dirs):
        out += sorted(glob.glob(os.path.join(d, f"{kind}_*.npz"))) + sorted(glob.glob(os.path.join(d, f"casadi_{kind}_*.npz")))
    return out
