"""Synthetic batches for the parity tests and the throughput harness (SURVEY.md section 8(d)).

Numeric settings follow `/root/reference/src/hippopt/turnkey_planners/humanoid_kinodynamic/
main_single_step_flat_ground.py:54-104` (config 3) and ``main_periodic_step.py`` (config 4);
instances differ in their initial state, references and evaluation point.
"""
from __future__ import annotations

import numpy as np

from .kino_layout import (COM, FD, F, H, NJ, NPT, NZ, P, PB, Q, QD, S, SD, U, V, VB, KinoLayout)
from .robot_model import RobotModel

FOOT_CORNERS = np.array([[0.116, 0.05, 0.0], [-0.116, 0.05, 0.0], [-0.116, -0.05, 0.0], [0.116, -0.05, 0.0]])
GRAVITY = np.array([0.0, 0.0, -9.80665, 0.0, 0.0, 0.0])


def kino_parameters(lay: KinoLayout, model: RobotModel, B: int, rng: np.random.Generator, spread: float = 1.0):
    """(B, n_p) parameter vectors in the reference's creation order (SURVEY.md Appendix B.2)."""
    po = lay.po
    N = lay.N
    p = np.zeros((B, lay.n_p))
    for k in range(N):
        for i in range(NPT):
            p[:, po.desc0 + 24 * k + 3 * i:po.desc0 + 24 * k + 3 * i + 3] = FOOT_CORNERS[i % 4]
    M = model.total_mass()
    p[:, po.mass] = M
    # initial / final state: feet flat at y = +-0.1, base above, forces = weight / 8 (mass-normalised)
    # on the stairs the robot starts in front of the first step edge (x = 0.225) and ends on it
    x_start = 0.15 if lay.st.terrain == "smooth_steps" else 0.0
    for base, dx in ((po.init, 0.0), (po.final, 0.3)):
        step = x_start + dx * rng.uniform(0.8, 1.2, B) * spread
        for i in range(NPT):
            y0 = 0.1 if i < 4 else -0.1
            o = base + po.st_pt(i, "p")
            p[:, o] = FOOT_CORNERS[i % 4, 0] + step
            p[:, o + 1] = FOOT_CORNERS[i % 4, 1] + y0
            p[:, o + 2] = 0.0
            o = base + po.st_pt(i, "f")
            p[:, o + 2] = 9.80665 / 8.0
            o = base + po.st_pt(i, "desc")
            p[:, o:o + 3] = FOOT_CORNERS[i % 4]
        p[:, base + po.ST_PB:base + po.ST_PB + 3] = np.array([0.0, 0.0, 0.75]) + np.stack(
            [step, np.zeros(B), np.zeros(B)], axis=1)
        qq = np.array([0.0, 0.0, 0.0, 1.0]) + 0.02 * spread * rng.normal(size=(B, 4))
        p[:, base + po.ST_Q:base + po.ST_Q + 4] = qq / np.linalg.norm(qq, axis=1, keepdims=True)
        p[:, base + po.ST_S:base + po.ST_S + NJ] = 0.05 * spread * rng.normal(size=(B, NJ))
        p[:, base + po.ST_COM:base + po.ST_COM + 3] = np.array([0.0, 0.0, 0.7]) + np.stack(
            [step, np.zeros(B), np.zeros(B)], axis=1)
    p[:, po.dt] = 0.1
    p[:, po.gravity:po.gravity + 6] = GRAVITY
    p[:, po.kt], p[:, po.k_bs], p[:, po.eps], p[:, po.mu] = 10.0, 40.0, 0.005, 0.3
    p[:, po.max_u:po.max_u + 3] = [2.0, 2.0, 5.0]
    p[:, po.max_fd:po.max_fd + 3] = 500.0
    p[:, po.max_L], p[:, po.min_com_h], p[:, po.min_feet_d], p[:, po.max_feet_h] = 5.0, 0.3, 0.1, 0.05
    p[:, po.max_s:po.max_s + NJ] = 1.5
    p[:, po.min_s:po.min_s + NJ] = -1.5
    p[:, po.max_sd:po.max_sd + NJ] = 2.0
    p[:, po.min_sd:po.min_sd + NJ] = -2.0
    for k in range(N):
        r = po.refs0 + 55 * k
        p[:, r + po.R_RATIO_L:r + po.R_RATIO_L + 4] = 0.25
        p[:, r + po.R_RATIO_R:r + po.R_RATIO_R + 4] = 0.25
        p[:, r + po.R_YAW_L] = 0.1 * spread * rng.normal(size=B)
        p[:, r + po.R_YAW_R] = 0.1 * spread * rng.normal(size=B)
        p[:, r + po.R_SWING] = 0.02
        p[:, r + po.R_CW:r + po.R_CW + 3] = [1.0, 1.0, 0.0]
        p[:, r + po.R_CC:r + po.R_CC + 3] = np.stack([0.3 * k / max(N - 1, 1) * np.ones(B), np.zeros(B), np.zeros(B)], 1)
        p[:, r + po.R_COMV:r + po.R_COMV + 3] = [0.1, 0.0, 0.0]
        for o in (po.R_FQ, po.R_BQ):
            qq = np.array([0.0, 0.0, 0.0, 1.0]) + 0.05 * spread * rng.normal(size=(B, 4))
            p[:, r + o:r + o + 4] = qq / np.linalg.norm(qq, axis=1, keepdims=True)
        p[:, r + po.R_BQV:r + po.R_BQV + 4] = 0.01 * spread * rng.normal(size=(B, 4))
        p[:, r + po.R_JR:r + po.R_JR + NJ] = 0.05 * spread * rng.normal(size=(B, NJ))
    if lay.st.terrain == "smooth_steps":
        # two smooth steps of `main_walking_on_stairs.py:18-28,397-403` (step_length 0.9, width 0.8), with
        # the step height randomised per instance in U(0.05, 0.15) (BASELINE config 5)
        L = 0.45
        height = rng.uniform(0.05, 0.15, B)
        tp = np.array([2 * L, 0.8, 0.0, 1.5 * L, 0.0, 0.9 * L, 0.8, 0.0, 2 * L, 0.0])
        p[:, po.terrain:po.terrain + 10] = tp
        p[:, po.terrain + 2] = height
        p[:, po.terrain + 7] = height
    elif lay.st.terrain == "tilted_steps":
        p[:, po.terrain:] = tilted_steps_sample(lay.st.n_terrain_params // 10, B, rng)
    return p


def tilted_steps_sample(K: int, B: int, rng: np.random.Generator) -> np.ndarray:
    """(B, 10 K) parameters of K rotated, raised and tilted steps that overlap around the origin, where the contact
    points of kino_points lie: per step (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z), a unit normal tilted by up to
    about 20 degrees."""
    tp = np.zeros((B, K, 10))
    tp[:, :, 0] = rng.uniform(0.6, 1.4, (B, K))
    tp[:, :, 1] = rng.uniform(0.5, 1.0, (B, K))
    tp[:, :, 2] = rng.uniform(0.02, 0.12, (B, K))
    tp[:, :, 3] = rng.uniform(-0.3, 0.3, (B, K))
    tp[:, :, 4] = rng.uniform(-0.2, 0.2, (B, K))
    tp[:, :, 5] = rng.uniform(-0.03, 0.03, (B, K))
    tp[:, :, 6] = rng.uniform(-0.6, 0.6, (B, K))
    n = np.concatenate([rng.uniform(-0.25, 0.25, (B, K, 2)), np.ones((B, K, 1))], axis=2)
    tp[:, :, 7:10] = n / np.linalg.norm(n, axis=2, keepdims=True)
    return tp.reshape(B, 10 * K)


def kino_points(lay: KinoLayout, p: np.ndarray, rng: np.random.Generator, noise: float = 1e-2):
    """Evaluation points: linear interpolation initial -> final state plus N(0, noise) (config 3)."""
    po = lay.po
    N = lay.N
    B = p.shape[0]
    x = np.zeros((B, lay.n_x))
    for k in range(N):
        a = k / max(N - 1, 1)
        z = x[:, NZ * k:NZ * (k + 1)]

        def blend(off, n):
            return (1 - a) * p[:, po.init + off:po.init + off + n] + a * p[:, po.final + off:po.final + off + n]

        for i in range(NPT):
            z[:, 15 * i + P:15 * i + P + 3] = blend(po.st_pt(i, "p"), 3)
            z[:, 15 * i + F:15 * i + F + 3] = blend(po.st_pt(i, "f"), 3)
        z[:, PB:PB + 3] = blend(po.ST_PB, 3)
        z[:, Q:Q + 4] = blend(po.ST_Q, 4)
        z[:, S:S + NJ] = blend(po.ST_S, NJ)
        z[:, COM:COM + 3] = blend(po.ST_COM, 3)
        z[:, VB] = 0.3 / (0.1 * N)
        z[:, H] = 0.3 / (0.1 * N)
    x += noise * rng.normal(size=x.shape)
    return x


def pose_batch(lay, model: RobotModel, B: int, seed: int = 1, noise: float = 0.05):
    """Pose-finder instances (BASELINE config 2, `humanoid_pose_finder/main.py:100-130`): references
    com = (0, 0, 0.7) + U(-0.05, 0.05) in xy, feet at (U(-0.15, 0.15), +-0.1, 0), identity quaternions, the
    reference joint configuration; evaluation points = references + N(0, noise)."""
    rng = np.random.default_rng(seed)
    po = lay.po
    p = np.zeros((B, lay.n_p))
    for i in range(NPT):
        p[:, po.desc0 + 3 * i:po.desc0 + 3 * i + 3] = FOOT_CORNERS[i % 4]
    p[:, po.mass] = model.total_mass()
    p[:, po.gravity:po.gravity + 6] = GRAVITY
    foot_x = rng.uniform(-0.15, 0.15, (B, 2))
    for i in range(NPT):
        o = po.ref + 9 * i
        p[:, o] = FOOT_CORNERS[i % 4, 0] + foot_x[:, i // 4]
        p[:, o + 1] = FOOT_CORNERS[i % 4, 1] + (0.1 if i < 4 else -0.1)
        p[:, o + 5] = 9.80665 / 8.0
        p[:, o + 6:o + 9] = FOOT_CORNERS[i % 4]
    p[:, po.ref + po.ST_PB:po.ref + po.ST_PB + 3] = [0.0, 0.0, 0.75]
    p[:, po.ref + po.ST_Q + 3] = 1.0
    s_ref = np.deg2rad([7, 0.12, -0.01, 12, 7, -12, 40.769, 12, 7, -12, 40.769, 5.76, 1.61, -0.31, -31.64, -20.52,
                        -1.52, 5.76, 1.61, -0.31, -31.64, -20.52, -1.52])
    p[:, po.ref + po.ST_S:po.ref + po.ST_S + NJ] = s_ref
    p[:, po.ref + po.ST_COM:po.ref + po.ST_COM + 3] = np.concatenate(
        [rng.uniform(-0.05, 0.05, (B, 2)), 0.7 * np.ones((B, 1))], axis=1)
    p[:, po.ref_fq + 3] = 1.0
    p[:, po.eps], p[:, po.mu] = 1e-4, 0.3
    p[:, po.max_s:po.max_s + NJ] = 1.5
    p[:, po.min_s:po.min_s + NJ] = -1.5
    x = np.zeros((B, lay.n_x))
    for i in range(NPT):
        x[:, 6 * i:6 * i + 6] = p[:, po.ref + 9 * i:po.ref + 9 * i + 6]
    x[:, 48:51] = p[:, po.ref + po.ST_PB:po.ref + po.ST_PB + 3]
    x[:, 51:55] = p[:, po.ref + po.ST_Q:po.ref + po.ST_Q + 4]
    x[:, 55:78] = p[:, po.ref + po.ST_S:po.ref + po.ST_S + NJ]
    x[:, 78:81] = p[:, po.ref + po.ST_COM:po.ref + po.ST_COM + 3]
    x += noise * rng.normal(size=x.shape)
    lam = rng.normal(size=(B, lay.m))
    return x, p, lam, np.ones(B)


def kino_batch(lay: KinoLayout, model: RobotModel, B: int, seed: int = 2, noise: float = 1e-2, spread: float = 1.0):
    """x, p, lam_g ~ N(0,1), sigma = 1 for B instances (seeded)."""
    rng = np.random.default_rng(seed)
    p = kino_parameters(lay, model, B, rng, spread)
    x = kino_points(lay, p, rng, noise)
    lam = rng.normal(size=(B, lay.m))
    sigma = np.ones(B)
    return x, p, lam, sigma


def standing_problem(lay: KinoLayout, model: RobotModel, pose: np.ndarray):
    """Kinodynamic "keep standing" OCPs from pose-finder solutions (SURVEY.md 8(f) f1/f3: the pose finder is
    what produces initial / final states in `main_periodic_step.py:192-327`).

    pose: (B, 81) pose-finder solutions [p_i, f_i (8 points), p_b, q, s, com].  Returns (p, x0): parameters
    whose initial state, final state and references are that pose, and the initial guess that repeats it at
    every knot with zero velocities -- feasible by construction (the pose finder enforces the static
    balance, the contact rows and the kinematic consistency the OCP asks for)."""
    po, N, B = lay.po, lay.N, pose.shape[0]
    p = kino_parameters(lay, model, B, np.random.default_rng(0), spread=0.0)
    for base in (po.init, po.final):
        for i in range(NPT):
            p[:, base + po.st_pt(i, "p"):base + po.st_pt(i, "p") + 3] = pose[:, 6 * i:6 * i + 3]
            p[:, base + po.st_pt(i, "f"):base + po.st_pt(i, "f") + 3] = pose[:, 6 * i + 3:6 * i + 6]
        p[:, base + po.ST_PB:base + po.ST_PB + 3] = pose[:, 48:51]
        p[:, base + po.ST_Q:base + po.ST_Q + 4] = pose[:, 51:55]
        p[:, base + po.ST_S:base + po.ST_S + NJ] = pose[:, 55:78]
        p[:, base + po.ST_COM:base + po.ST_COM + 3] = pose[:, 78:81]
    centroid = np.stack([pose[:, 6 * i:6 * i + 3] for i in range(NPT)], axis=0).mean(axis=0)
    for k in range(N):
        r = po.refs0 + 55 * k
        p[:, r + po.R_CC:r + po.R_CC + 3] = centroid
        p[:, r + po.R_COMV:r + po.R_COMV + 3] = 0.0
        p[:, r + po.R_SWING] = 0.0
        p[:, r + po.R_YAW_L] = p[:, r + po.R_YAW_R] = 0.0
        p[:, r + po.R_BQ:r + po.R_BQ + 4] = pose[:, 51:55]
        p[:, r + po.R_FQ:r + po.R_FQ + 4] = [0.0, 0.0, 0.0, 1.0]
        p[:, r + po.R_BQV:r + po.R_BQV + 4] = 0.0
        p[:, r + po.R_JR:r + po.R_JR + NJ] = pose[:, 55:78]
    x0 = np.zeros((B, lay.n_x))
    for k in range(N):
        z = x0[:, NZ * k:NZ * (k + 1)]
        for i in range(NPT):
            z[:, 15 * i + P:15 * i + P + 3] = pose[:, 6 * i:6 * i + 3]
            z[:, 15 * i + F:15 * i + F + 3] = pose[:, 6 * i + 3:6 * i + 6]
        z[:, PB:PB + 3] = pose[:, 48:51]
        z[:, Q:Q + 4] = pose[:, 51:55]
        z[:, S:S + NJ] = pose[:, 55:78]
        z[:, COM:COM + 3] = pose[:, 78:81]
    return p, x0


def transfer_problem(lay: KinoLayout, model: RobotModel, pose_a: np.ndarray, pose_b: np.ndarray):
    """OCPs that go from pose A to pose B (SURVEY.md 8(f) f3): initial state A, final state B (use a layout with
    ``final_state_constraint``), references and initial guess interpolated linearly knot by knot -- the role of
    `humanoid_state_interpolator` (`robot_planning/utilities/interpolators.py:396-448`) for states without a
    contact-phase change (the quaternion is interpolated linearly and left to the unit-norm row, not slerped).
    The guess has zero velocities, i.e. it violates the integrator rows by O(|B - A| / N)."""
    pa, xa = standing_problem(lay, model, pose_a)
    pb, xb = standing_problem(lay, model, pose_b)
    po, N = lay.po, lay.N
    n_state = po.ST_COM + 3  # one state block: points, base, joints, com
    pa[:, po.final:po.final + n_state] = pb[:, po.final:po.final + n_state]
    for k in range(N):
        w = k / max(N - 1, 1)
        r = po.refs0 + 55 * k
        pa[:, r:r + 55] = (1 - w) * pa[:, r:r + 55] + w * pb[:, r:r + 55]
        xa[:, NZ * k:NZ * (k + 1)] = (1 - w) * xa[:, NZ * k:NZ * (k + 1)] + w * xb[:, NZ * k:NZ * (k + 1)]
    return pa, xa
