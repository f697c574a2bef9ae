"""Initial states, final states and initial guesses for a batch of periodic-step plans, on the device
(SURVEY.md 8(f) row f3).  The batched counterpart of the set-up part of
/root/reference/src/hippopt/turnkey_planners/humanoid_kinodynamic/main_periodic_step.py:

* contact phase guesses of a step of length L per instance (:365-412),
* three pose-finder solves per instance -- initial, middle and final double-support keyframes
  (compute_state / compute_initial_state / compute_middle_state / compute_final_state, :192-327) -- as ONE batch of
  3 B instances of the interior-point driver (ipsolver.py) over the pose-finder evaluator,
* `humanoid_state_interpolator` over the two halves (:433-451) written straight into the decision vectors
  (interpolators.py -> csrc/interp.cu),
* the references of get_references (:330-352) and the initial / final state parameters (:470-478).

`stairs_step_guess` builds the same set-up for BASELINE config 5 (walking on stairs): the keyframe poses are solved on
the smooth-step terrain (pose-finder evaluator with ``terrain="smooth_steps"``), and the contacts land on the first
tread.  `ramp_step_guess` does the same for a step onto a ramp (``terrain="tilted_steps"``, one tilted step).

Everything numeric runs on the GPU; the per-instance Python loop of the reference (one IPOPT solve after the other)
is gone.  How far the interior-point driver gets on the plans built here (some converge, many do not) is recorded
in DESIGN.md section 9, row (f), and profiles/r01/solver_v11.txt."""
from __future__ import annotations

import dataclasses

import numpy as np
import torch

from .interpolators import FeetContactPhasesDescriptor, FootContactPhaseDescriptor, humanoid_state_interpolator
from .ipsolver import BatchedInteriorPoint
from .kino_layout import NJ, NPT
from .workloads import FOOT_CORNERS, GRAVITY, kino_parameters

DESIRED_JOINTS_DEG = [7, 0.12, -0.01, 12, 7, -12, 40.769, 12, 7, -12, 40.769, 5.76, 1.61, -0.31, -31.64, -20.52, -1.52,
                      5.76, 1.61, -0.31, -31.64, -20.52, -1.52]  # main_periodic_step.py:199-225


def periodic_step_phases(step_length: np.ndarray, horizon_time: float, foot_y: float = 0.1,
                         swing_height: float = 0.05, force_z: float = 100.0) -> FeetContactPhasesDescriptor:
    """main_periodic_step.py:365-412 with a step length per instance (the reference uses 0.6 for ergoCub)."""
    L = np.asarray(step_length, dtype=np.float64).reshape(-1)
    B = L.shape[0]

    def pos(x, y, z):
        return np.stack([x, np.full(B, y), np.full(B, z)], axis=1)

    return _left_then_right(pos(0 * L, foot_y, 0.0), pos(L / 2, foot_y, swing_height), pos(L, foot_y, 0.0),
                            pos(L / 2, -foot_y, 0.0), pos(L, -foot_y, swing_height), pos(1.5 * L, -foot_y, 0.0),
                            horizon_time, force_z)


def _left_then_right(l0, l_mid, l1, r0, r_mid, r1, T, force_z, q1=None):
    """Two contact phases per foot, (B, 3) positions: the left foot swings from l0 over l_mid to l1 in (T/6, T/3), then
    the right foot from r0 over r_mid to r1 in (2T/3, 5T/6) (main_periodic_step.py:365-412).  Identity rotations, except
    that q1 (xyzw, (4,) or (B, 4)), if given, is the rotation of both feet at their landing (and mid-swing) poses."""
    ident = np.array([0.0, 0.0, 0.0, 1.0])
    q1 = ident if q1 is None else q1

    def phase(p, mid, act, dea, q):
        return FootContactPhaseDescriptor(position=p, quaternion_xyzw=q, mid_swing_position=mid,
                                          mid_swing_quaternion_xyzw=None if mid is None else q1,
                                          force=np.array([0.0, 0.0, force_z]), activation_time=act, deactivation_time=dea)

    return FeetContactPhasesDescriptor(
        left=[phase(l0, l_mid, None, T / 6.0, ident), phase(l1, None, T / 3.0, None, q1)],
        right=[phase(r0, r_mid, None, T * 2.0 / 3.0, ident), phase(r1, None, T * 5.0 / 6.0, None, q1)])


def pose_problem(lay, model, left_position: np.ndarray, right_position: np.ndarray, com_height: float = 0.7,
                 left_rotation: np.ndarray | None = None, right_rotation: np.ndarray | None = None):
    """Pose-finder references of compute_state (main_periodic_step.py:192-258) for feet at the given positions
    (identity rotations, or the (B, 3, 3) rotations given): contact points from the foot transforms, CoM com_height
    above the middle of the feet, identity base / frame quaternions, the desired joint configuration.  Returns
    (x guess, p); on a smooth-step terrain the caller fills the terrain parameters."""
    po = lay.po
    B = left_position.shape[0]
    rot = [left_rotation, right_rotation]
    p = np.zeros((B, lay.n_p))
    for i in range(NPT):
        p[:, po.desc0 + 3 * i:po.desc0 + 3 * i + 3] = FOOT_CORNERS[i % 4]
    p[:, po.mass] = model.total_mass()
    p[:, po.gravity:po.gravity + 6] = GRAVITY
    feet = (left_position, right_position)
    for i in range(NPT):
        o = po.ref + 9 * i
        R = rot[i // 4]
        p[:, o:o + 3] = feet[i // 4] + (FOOT_CORNERS[i % 4] if R is None else R @ FOOT_CORNERS[i % 4])
        p[:, o + 5] = 9.80665 / 8.0
        p[:, o + 6:o + 9] = FOOT_CORNERS[i % 4]
    com = (left_position + right_position) / 2.0
    com[:, 2] += com_height
    p[:, po.ref + po.ST_PB:po.ref + po.ST_PB + 3] = com + [0.0, 0.0, 0.05]
    p[:, po.ref + po.ST_Q + 3] = 1.0
    p[:, po.ref + po.ST_S:po.ref + po.ST_S + NJ] = np.deg2rad(DESIRED_JOINTS_DEG)
    p[:, po.ref + po.ST_COM:po.ref + po.ST_COM + 3] = com
    p[:, po.ref_fq + 3] = 1.0
    p[:, po.eps], p[:, po.mu] = 1e-4, 0.3
    p[:, po.max_s:po.max_s + NJ] = 1.5
    p[:, po.min_s:po.min_s + NJ] = -1.5
    x = np.zeros((B, lay.n_x))
    for i in range(NPT):
        x[:, 6 * i:6 * i + 6] = p[:, po.ref + 9 * i:po.ref + 9 * i + 6]
    x[:, 48:81] = p[:, po.ref + po.ST_PB:po.ref + po.ST_COM + 3]
    return x, p


def state_blocks(pose: torch.Tensor) -> torch.Tensor:
    """(B, 81) pose-finder solutions [8 x (p, f), p_b, q, s, com] -> (B, 105) state blocks [8 x (p, f, descriptor), ...]."""
    B = pose.shape[0]
    corners = torch.as_tensor(np.tile(FOOT_CORNERS, (2, 1)), dtype=pose.dtype, device=pose.device)
    pts = torch.cat([pose[:, :48].reshape(B, NPT, 6), corners.expand(B, NPT, 3)], dim=2).reshape(B, 72)
    return torch.cat([pts, pose[:, 48:81]], dim=1).contiguous()


@dataclasses.dataclass
class PeriodicStepGuess:
    parameters: np.ndarray  # (B, n_p) of the kinodynamic NLP
    x0: torch.Tensor  # (B, n_x) initial guess on the device
    ok: torch.Tensor  # (B,) all three keyframe poses converged
    keyframes: torch.Tensor  # (3, B, 105) initial, middle, final state blocks
    pose_iterations: torch.Tensor  # (3 B,)


def periodic_step_guess(model, pose_evaluator, kino_evaluator, step_length: np.ndarray, tol: float = 1e-8,
                        max_iter: int = 300, force_z: float = 100.0, mass_normalised: bool = False) -> PeriodicStepGuess:
    """main_periodic_step.py:365-478 for a batch of step lengths (see the module docstring).  force_z: the planned
    contact force of the phases, 100 N per point in the reference's main.  The planner divides every force of the
    guess by the robot's mass before it reaches the NLP (`planner.py:932-980`, `_apply_mass_regularization`, called
    from `set_initial_guess`): mass_normalised=True does the same, so that force_z = 100 IS the reference's guess."""
    if mass_normalised:
        force_z = force_z / float(model.total_mass())
    L = np.asarray(step_length, dtype=np.float64).reshape(-1)
    phases = periodic_step_phases(L, kino_evaluator.layout.N * STEP_DT, force_z=force_z)
    centroid = np.stack([L / 2.0, np.zeros_like(L), np.zeros_like(L)], axis=1)  # 0.3 for the reference's 0.6 m step
    return _keyframe_plan(model, pose_evaluator, kino_evaluator, phases, centroid, None, tol, max_iter)


STEP_DT = 0.1


def _keyframe_plan(model, pose_evaluator, kino_evaluator, phases, centroid, terrain, tol, max_iter) -> PeriodicStepGuess:
    """The part periodic_step_guess and stairs_step_guess share: the initial / middle / final keyframe poses at the
    phases' contact positions as one pose-finder batch, the interpolated guess, and the kinodynamic parameters
    (initial / final states and the references of get_references with the contact centroid ``centroid`` (B, 3)).
    ``terrain``: (B, n) terrain parameters of both problems, or None on the planar terrain."""
    lay, pl = kino_evaluator.layout, pose_evaluator.layout
    N, po = lay.N, lay.po
    B = centroid.shape[0]
    dev = torch.device("cuda", torch.cuda.current_device())
    dt = STEP_DT
    # keyframes: (left phase, right phase) of compute_initial_state / compute_middle_state / compute_final_state
    lp = np.concatenate([phases.left[0].position, phases.left[1].position, phases.left[1].position])
    rp = np.concatenate([phases.right[0].position, phases.right[0].position, phases.right[1].position])

    def rotations(ph):  # (B, 3, 3) foot rotation of a phase, or None when it is the identity
        q = np.broadcast_to(np.asarray(ph.quaternion_xyzw, dtype=np.float64), (B, 4))
        if np.all(q == [0.0, 0.0, 0.0, 1.0]):
            return None
        return _rotation_xyzw(q)

    lr = [rotations(phases.left[0]), rotations(phases.left[1]), rotations(phases.left[1])]
    rr = [rotations(phases.right[0]), rotations(phases.right[0]), rotations(phases.right[1])]
    ident = np.broadcast_to(np.eye(3), (B, 3, 3))
    lrot = None if all(r is None for r in lr) else np.concatenate([ident if r is None else r for r in lr])
    rrot = None if all(r is None for r in rr) else np.concatenate([ident if r is None else r for r in rr])
    xq, pq = pose_problem(pl, model, lp, rp, left_rotation=lrot, right_rotation=rrot)
    if terrain is not None:
        pq[:, pl.po.terrain:pl.po.terrain + terrain.shape[1]] = np.tile(terrain, (3, 1))
    lb, ub = pose_evaluator.bounds(pq)
    out = BatchedInteriorPoint(pose_evaluator, tol=tol, max_iter=max_iter).solve(
        torch.tensor(xq, device=dev), torch.tensor(pq, device=dev), lb, ub)  # OptiFailure if no keyframe pose converges at all
    key = state_blocks(out.values).view(3, B, 105)
    ok = out.success.view(3, B).all(dim=0)

    x0 = torch.zeros((B, lay.n_x), dtype=torch.float64, device=dev)
    half = N // 2
    humanoid_state_interpolator(key[0], key[1], phases, half, dt, x_out=x0, states_out=False)
    second = humanoid_state_interpolator(key[1], key[2], phases, N - half, dt, t0=half * dt, x_out=x0, knot0=half)
    first = humanoid_state_interpolator(key[0], key[1], phases, half, dt)
    guess = torch.cat([first, second], dim=1).cpu().numpy()  # (B, N, 105): the joint references below

    p = kino_parameters(lay, model, B, np.random.default_rng(0), spread=0.0)
    if terrain is not None:
        p[:, po.terrain:po.terrain + terrain.shape[1]] = terrain
    k0, k2 = key[0].cpu().numpy(), key[2].cpu().numpy()
    n_state = po.ST_COM + 3
    p[:, po.init:po.init + n_state] = k0
    p[:, po.final:po.final + n_state] = k2
    for k in range(N):
        r = po.refs0 + 55 * k  # get_references, main_periodic_step.py:330-352
        p[:, r + po.R_CW:r + po.R_CW + 3] = [100.0, 100.0, 10.0]
        p[:, r + po.R_CC:r + po.R_CC + 3] = centroid
        p[:, r + po.R_COMV:r + po.R_COMV + 3] = [0.1, 0.0, 0.0]
        p[:, r + po.R_YAW_L] = p[:, r + po.R_YAW_R] = 0.0
        p[:, r + po.R_FQ:r + po.R_FQ + 4] = [0.0, 0.0, 0.0, 1.0]
        p[:, r + po.R_BQ:r + po.R_BQ + 4] = [0.0, 0.0, 0.0, 1.0]
        p[:, r + po.R_BQV:r + po.R_BQV + 4] = 0.0
        p[:, r + po.R_JR:r + po.R_JR + NJ] = guess[:, k, 79:79 + NJ]
    return PeriodicStepGuess(parameters=p, x0=x0, ok=ok, keyframes=key, pose_iterations=out.iterations)


# the stairs of workloads.kino_parameters (main_walking_on_stairs.py:18-28, 397-403): two smooth steps, the first tread
# at height h for x in (0.225, 0.6975), the second at 2 h beyond; each edge's transition band is about 2 cm wide
def stairs_terrain(step_height: np.ndarray) -> np.ndarray:
    """(B, 10) terrain parameters (l, w, height, ox, oy) x 2 of the stairs with the step height h per instance."""
    h = np.asarray(step_height, dtype=np.float64).reshape(-1)
    L = 0.45
    tp = np.tile([2 * L, 0.8, 0.0, 1.5 * L, 0.0, 0.9 * L, 0.8, 0.0, 2 * L, 0.0], (h.shape[0], 1))
    tp[:, 2] = tp[:, 7] = h
    return tp


def stairs_step_guess(model, pose_evaluator, kino_evaluator, step_height: np.ndarray, tol: float = 1e-8,
                      max_iter: int = 300, force_z: float = 100.0, mass_normalised: bool = False,
                      start_x: float = 0.0, tread_x: float = 0.45, foot_y: float = 0.1,
                      swing_height: float = 0.05) -> PeriodicStepGuess:
    """BASELINE config 5 (walking on stairs, N = 50, dt = 0.1): the batched counterpart of periodic_step_guess on the
    stairs of `stairs_terrain`, with the step height h per instance.  The robot starts with both feet on the ground
    centred at x = start_x (every foot corner, +-0.116 m, clear of the first edge's transition band), steps with the
    left foot onto the first tread (centred at x = tread_x, clear of both of its edges), then with the right foot.

    * keyframes: initial (both feet on the ground), middle (left foot on the first tread), final (both feet on the first
      tread), three pose-finder solves per instance as ONE batch of 3 B on the smooth-terrain pose evaluator;
    * point references and contact phases: the z of every point is the height of the tread it lands on, the mid-swing
      height is the higher tread plus swing_height;
    * guess and references as periodic_step_guess (interpolation over both halves, get_references with the contact
      centroid halfway between start and tread, at half the step height).

    UNPINNED: the reference's stairs main (main_walking_on_stairs.py) is available here only through the lines SURVEY.md
    cites (terrain, horizon and solver options); this keyframe placement is this project's own, not a restatement."""
    if mass_normalised:
        force_z = force_z / float(model.total_mass())
    h = np.asarray(step_height, dtype=np.float64).reshape(-1)
    B = h.shape[0]
    if pose_evaluator.layout.st.terrain != "smooth_steps" or kino_evaluator.layout.st.terrain != "smooth_steps":
        raise ValueError("stairs_step_guess: both evaluators must be posed on the smooth steps")

    def pos(x, y, z):
        return np.stack([np.full(B, x), np.full(B, y), z], axis=1)

    zero = np.zeros(B)
    mid_x = 0.5 * (start_x + tread_x)
    phases = _left_then_right(pos(start_x, foot_y, zero), pos(mid_x, foot_y, h + swing_height), pos(tread_x, foot_y, h),
                              pos(start_x, -foot_y, zero), pos(mid_x, -foot_y, h + swing_height),
                              pos(tread_x, -foot_y, h), kino_evaluator.layout.N * STEP_DT, force_z)
    centroid = pos(mid_x, 0.0, 0.5 * h)
    return _keyframe_plan(model, pose_evaluator, kino_evaluator, phases, centroid, stairs_terrain(h), tol, max_iter)


def _rotation_xyzw(q: np.ndarray) -> np.ndarray:
    """(B, 4) unit quaternions (x, y, z, w) -> (B, 3, 3) rotation matrices."""
    x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    return np.stack([
        np.stack([1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)], axis=1),
        np.stack([2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)], axis=1),
        np.stack([2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)], axis=1)], axis=1)


def tilted_steps_terrain(length, width, height, origin, yaw=0.0, normal=(0.0, 0.0, 1.0)) -> np.ndarray:
    """(B, 10 K) parameters of K general smooth steps (``terrain="tilted_steps"``), the arguments of
    `SmoothTerrain.step` (smooth_terrain.py:235-336) per step: length l, width w, height, origin (ox, oy, oz), yaw and
    the normal (n_x, n_y, n_z) of the tilted top.  Each argument is a scalar, a (K,) or (B, K) array (origin and normal:
    (3,), (K, 3) or (B, K, 3)); a leading batch dimension B broadcasts.  The normal is taken as given (the reference does
    not normalise it either); l, w > 0 and n_z > 0 are required."""
    lw = np.asarray(length, dtype=np.float64)
    K = 1 if lw.ndim == 0 else lw.shape[-1]

    def scalars(a):
        a = np.asarray(a, dtype=np.float64)
        return np.atleast_2d(a.reshape(-1, K) if a.ndim else np.full((1, K), float(a)))

    def vectors(a):
        a = np.asarray(a, dtype=np.float64)
        return a.reshape(1, 1, 3) if a.ndim == 1 else (a.reshape(1, K, 3) if a.ndim == 2 else a)

    cols = [scalars(length), scalars(width), scalars(height), vectors(origin), scalars(yaw), vectors(normal)]
    B = max(c.shape[0] for c in cols)
    tp = np.zeros((B, K, 10))
    tp[:, :, 0], tp[:, :, 1], tp[:, :, 2] = (np.broadcast_to(c, (B, K)) for c in cols[:3])
    tp[:, :, 3:6] = np.broadcast_to(cols[3], (B, K, 3))
    tp[:, :, 6] = np.broadcast_to(cols[4], (B, K))
    tp[:, :, 7:10] = np.broadcast_to(cols[5], (B, K, 3))
    if not np.all(np.isfinite(tp)):
        raise ValueError("tilted_steps_terrain: non-finite parameter")
    if np.any(tp[:, :, 0] <= 0.0) or np.any(tp[:, :, 1] <= 0.0):
        raise ValueError("tilted_steps_terrain: length and width must be positive")
    if np.any(tp[:, :, 9] <= 0.0):
        raise ValueError("tilted_steps_terrain: the normal's z component must be positive")
    return tp.reshape(B, 10 * K)


# the ramp of ramp_step_guess: one smooth step of length RAMP_LENGTH whose top rises along +x with the slope s (rise
# over run), its low edge (at height 0) at x = RAMP_START, its high edge at height s RAMP_LENGTH
RAMP_START, RAMP_LENGTH, RAMP_WIDTH = 0.225, 2.0, 0.8


def ramp_terrain(slope: np.ndarray) -> np.ndarray:
    """(B, 10) tilted_steps parameters of the ramp with the slope s (rise over run) per instance."""
    s = np.asarray(slope, dtype=np.float64).reshape(-1)
    n = np.stack([-s, np.zeros_like(s), np.ones_like(s)], axis=1) / np.sqrt(1.0 + s * s)[:, None]
    return tilted_steps_terrain(RAMP_LENGTH, RAMP_WIDTH, s[:, None] * (0.5 * RAMP_LENGTH),
                                [RAMP_START + 0.5 * RAMP_LENGTH, 0.0, 0.0], 0.0, n[:, None, :])


def ramp_step_guess(model, pose_evaluator, kino_evaluator, slope: np.ndarray, tol: float = 1e-8, max_iter: int = 300,
                    force_z: float = 100.0, mass_normalised: bool = False, start_x: float = 0.0,
                    tread_x: float = 0.5, foot_y: float = 0.1, swing_height: float = 0.05) -> PeriodicStepGuess:
    """The ramp counterpart of stairs_step_guess (N = 50, dt = 0.1): a step onto the ramp of `ramp_terrain` with the
    slope s per instance, on evaluators posed on ``terrain="tilted_steps"`` with one step.  The robot starts with both
    feet flat on the ground centred at x = start_x (every foot corner clear of the ramp's low edge at RAMP_START), steps
    with the left foot onto the slope (centred at x = tread_x), then with the right foot.

    * keyframes: initial (both feet on the ground), middle (left foot on the slope), final (both feet on the slope),
      three pose-finder solves per instance as ONE batch of 3 B; the feet on the slope are pitched to it (rotation
      about y by -atan s) and their centres lie on the slope's surface;
    * guess and references as stairs_step_guess (contact centroid halfway between start and tread, at half the tread
      height).

    UNPINNED: the reference's ramp main is available here only through the terrain SURVEY.md A.10 cites; this keyframe
    placement is this project's own, not a restatement."""
    if mass_normalised:
        force_z = force_z / float(model.total_mass())
    s = np.asarray(slope, dtype=np.float64).reshape(-1)
    B = s.shape[0]
    for ev in (pose_evaluator, kino_evaluator):
        if ev.layout.st.terrain != "tilted_steps" or ev.layout.st.n_terrain_params != 10:
            raise ValueError("ramp_step_guess: both evaluators must be posed on tilted_steps with one step")

    def pos(x, y, z):
        return np.stack([np.full(B, x), np.full(B, y), z], axis=1)

    zero = np.zeros(B)
    top = s * (tread_x - RAMP_START)  # surface height under the tread's centre
    mid_x = 0.5 * (start_x + tread_x)
    half = -0.5 * np.arctan(s)  # pitch about y that lifts the toe onto the slope
    q1 = np.stack([zero, np.sin(half), zero, np.cos(half)], axis=1)
    phases = _left_then_right(pos(start_x, foot_y, zero), pos(mid_x, foot_y, top + swing_height),
                              pos(tread_x, foot_y, top), pos(start_x, -foot_y, zero),
                              pos(mid_x, -foot_y, top + swing_height), pos(tread_x, -foot_y, top),
                              kino_evaluator.layout.N * STEP_DT, force_z, q1=q1)
    centroid = pos(mid_x, 0.0, 0.5 * top)
    return _keyframe_plan(model, pose_evaluator, kino_evaluator, phases, centroid, ramp_terrain(s), tol, max_iter)


def single_step_problem(model, pose_evaluator, kino_evaluator, step_length: np.ndarray, tol: float = 1e-8,
                        max_iter: int = 300) -> PeriodicStepGuess:
    """BASELINE config 3, main_single_step_flat_ground.py:188-356, for a batch of step lengths: the initial state
    (feet side by side, `compute_initial_state` :188-262) and the final state (right foot one step ahead, CoM half
    a step ahead, `compute_final_state` :265-338) from 2 B pose-finder solves, and the references of
    `get_references` (:341-356: contact centroid one step ahead with weights (100, 100, 10), joint regularisation
    towards the final joints, CoM velocity 0.1 m/s forward), scaled from the main's 0.3 m step to L.

    The main hands IPOPT no initial guess (the planner's default variables); here the guess holds the initial state
    over the horizon with zero velocities -- the same "standing" start in the layout of the decision vector."""
    lay, pl = kino_evaluator.layout, pose_evaluator.layout
    N, po = lay.N, lay.po
    L = np.asarray(step_length, dtype=np.float64).reshape(-1)
    B = L.shape[0]
    dev = torch.device("cuda", torch.cuda.current_device())
    zero = np.zeros(B)

    def pos(x, y):
        return np.stack([x, np.full(B, y), zero], axis=1)

    lp = np.concatenate([pos(zero, 0.1), pos(zero, 0.1)])
    rp = np.concatenate([pos(zero, -0.1), pos(L, -0.1)])
    xq, pq = pose_problem(pl, model, lp, rp)
    lb, ub = pose_evaluator.bounds(pq)
    out = BatchedInteriorPoint(pose_evaluator, tol=tol, max_iter=max_iter).solve(
        torch.tensor(xq, device=dev), torch.tensor(pq, device=dev), lb, ub)
    key = state_blocks(out.values).view(2, B, 105)
    ok = out.success.view(2, B).all(dim=0)
    k0, k2 = key[0].cpu().numpy(), key[1].cpu().numpy()
    p = kino_parameters(lay, model, B, np.random.default_rng(0), spread=0.0)
    n_state = po.ST_COM + 3
    p[:, po.init:po.init + n_state] = k0
    p[:, po.final:po.final + n_state] = k2
    for k in range(N):
        r = po.refs0 + 55 * k
        p[:, r + po.R_CW:r + po.R_CW + 3] = [100.0, 100.0, 10.0]
        p[:, r + po.R_CC] = L
        p[:, r + po.R_CC + 1:r + po.R_CC + 3] = 0.0
        p[:, r + po.R_COMV:r + po.R_COMV + 3] = [0.1, 0.0, 0.0]
        p[:, r + po.R_YAW_L] = p[:, r + po.R_YAW_R] = 0.0
        p[:, r + po.R_FQ:r + po.R_FQ + 4] = [0.0, 0.0, 0.0, 1.0]
        p[:, r + po.R_BQ:r + po.R_BQ + 4] = [0.0, 0.0, 0.0, 1.0]
        p[:, r + po.R_BQV:r + po.R_BQV + 4] = 0.0
        p[:, r + po.R_JR:r + po.R_JR + NJ] = k2[:, po.ST_S:po.ST_S + NJ]
    # guess: the initial state at every knot (points p, f; base; joints; CoM), velocities and momentum zero
    from .kino_layout import COM, F, NZ, P, PB, Q, S

    x0 = np.zeros((B, lay.n_x))
    for k in range(N):
        z = x0[:, NZ * k:NZ * (k + 1)]
        for i in range(NPT):
            z[:, 15 * i + P:15 * i + P + 3] = k0[:, 9 * i:9 * i + 3]
            z[:, 15 * i + F:15 * i + F + 3] = k0[:, 9 * i + 3:9 * i + 6]
        z[:, PB:PB + 3] = k0[:, po.ST_PB:po.ST_PB + 3]
        z[:, Q:Q + 4] = k0[:, po.ST_Q:po.ST_Q + 4]
        z[:, S:S + NJ] = k0[:, po.ST_S:po.ST_S + NJ]
        z[:, COM:COM + 3] = k0[:, po.ST_COM:po.ST_COM + 3]
    return PeriodicStepGuess(parameters=p, x0=torch.tensor(x0, device=dev), ok=ok,
                             keyframes=torch.stack([key[0], key[1], key[1]]), pose_iterations=out.iterations)
