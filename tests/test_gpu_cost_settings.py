"""The evaluation kernels under non-default cost settings, against the CPU oracle built with the same settings.

The weights, the yaw points and the foot and frame-cost bodies are runtime data of the kernels (the HB_KD_* / HB_KI_*
tables of include/hippopt_b200.h), and the closed forms of the contact and kinematics kernels use them directly.  At
the default settings several mistakes cancel: the CoM-velocity multiplier is 1, two pose weights are equal, the joint
weights repeat in groups, and only one geometry exists.  So these tests use settings in which no two numbers are equal
and none is 1 (tests_support.distinct_cost_settings), every cost term on its own, other yaw points, feet and frame-cost
bodies, and the zero weights of the reference's own configurations.

Comparison: oracle/parity.check_all at 1e-10.  With every multiplier but one at zero and lam_g = 0, f, grad_f and hess_l
are that one term, so each term is checked at 1e-10 of its own size instead of the size of the largest term."""
import itertools

import numpy as np
import pytest
import torch

from tests_support import KINO_MULTIPLIERS, POSE_MULTIPLIERS, distinct_cost_settings, only_term, oracle_settings

pytestmark = pytest.mark.gpu

RTOL = 1e-10
SIGMA3 = np.array([0.0, 0.37, 3.5])
# two instances: the first with lam_g = 0 (hess_l is the cost alone), the second with random lam_g
SIGMA2 = np.array([0.37, 2.0])


def dev():
    return torch.device("cuda:0")


def run(ev, x, p, lam, sigma, mask=None):
    from hippopt_b200.evaluator import ALL

    t = [torch.tensor(np.ascontiguousarray(a), device=dev()) for a in (x, p, lam, sigma)]
    out = ev.eval(ALL if mask is None else mask, *t)
    torch.cuda.synchronize()
    return {k: v.cpu().numpy().copy() for k, v in out.items()}


def kino(model, N, fin=False, per=False, smooth=False, **settings):
    """(evaluator, oracle NLP) of the kinodynamic problem under the same settings."""
    from hippopt_b200.evaluator import KinoEvaluator
    from hippopt_b200.kino_layout import KinoSettings
    from oracle import expressions as ex
    from oracle import kinodynamic as kd

    terrain = dict(terrain="smooth_steps", n_terrain_params=10) if smooth else {}
    st = KinoSettings(horizon=N, final_state_constraint=fin, periodicity_constraint=per, **terrain, **settings)
    extra = dict(terrain=ex.TwoSmoothSteps(), terrain_params=10) if smooth else {}
    nlp, _ = kd.build(model, oracle_settings(kd.Settings, st, **extra))
    return KinoEvaluator(model, st), nlp


def pose(model, **settings):
    from hippopt_b200.evaluator import PoseEvaluator
    from hippopt_b200.pose_layout import PoseSettings
    from oracle import pose_finder as pf

    st = PoseSettings(**settings)
    nlp, _ = pf.build(model, oracle_settings(pf.Settings, st))
    return PoseEvaluator(model, st), nlp


def inputs(ev, model, B, seed):
    from hippopt_b200.workloads import kino_batch, pose_batch

    if ev.layout.__class__.__name__ == "PoseLayout":
        return pose_batch(ev.layout, model, B, seed=seed, noise=0.2)
    smooth = ev.settings.terrain != "planar"
    return kino_batch(ev.layout, model, B, seed=seed, noise=0.05 if smooth else 0.2, spread=1.0 if smooth else 2.0)


def two_instances(ev, model, seed):
    """x, p of two instances, lam_g = 0 for the first and random for the second, sigma = SIGMA2."""
    x, p, lam, _ = inputs(ev, model, 2, seed)
    lam[0] = 0.0
    return x, p, lam, SIGMA2.copy()


def on_layout_pattern(ev, nlp, ref_hess):
    """The oracle's Hessian values spread onto the layout's pattern, and the layout entries the oracle does not have
    (CasADi-style simplification of 0 * expr drops them)."""
    n = ev.n_x
    hc, hr = ev.hess_sparsity()
    lay_keys = np.repeat(np.arange(n), np.diff(hc)) * n + hr
    okeys = nlp.hess_structure()[3]
    at = np.searchsorted(lay_keys, okeys)
    assert np.array_equal(lay_keys[np.minimum(at, len(lay_keys) - 1)], okeys), "oracle entry outside the layout"
    full = np.zeros((ref_hess.shape[0], len(lay_keys)), dtype=ref_hess.dtype)
    full[:, at] = ref_hess
    dropped = np.setdiff1d(np.arange(len(lay_keys)), at)
    return full, dropped


def compare(ev, nlp, x, p, lam, sigma, longdouble=False, out=None, label=""):
    """Every output of the kernels against the oracle; returns (kernel outputs, worst relative error per output)."""
    from oracle import parity

    assert np.array_equal(ev.jac_sparsity()[0], nlp.jac_structure()[0])
    assert np.array_equal(ev.jac_sparsity()[1], nlp.jac_structure()[1])
    out = run(ev, x, p, lam, sigma) if out is None else out
    ref = parity.reference_outputs(nlp, x, p, lam, sigma, dtype=np.longdouble if longdouble else np.float64)
    for k, r in ref.items():
        assert np.isfinite(r).all() and np.isfinite(out[k]).all(), k
    ref["hess"], dropped = on_layout_pattern(ev, nlp, ref["hess"])
    if len(dropped):
        assert np.all(out["hess"][:, dropped] == 0.0), "kernel value at an entry the oracle proves zero"
    worst = parity.check_all(out, ref, ev.jac_sparsity(), ev.hess_sparsity(), x, rtol=RTOL)
    print(f"{label} worst relative errors:", {k: f"{v:.2e}" for k, v in worst.items()},
          f"({len(dropped)} dropped entries)" if len(dropped) else "")
    return out, worst


# ------------------------------------------------------------------------------------------------ a. distinct settings
CASES_A = {"kino_n3_final_periodic": dict(N=3, fin=True, per=True), "kino_n2": dict(N=2),
           "smooth_n3_final": dict(N=3, fin=True, smooth=True), "pose": None}


@pytest.mark.parametrize("case", list(CASES_A))
def test_distinct_settings_against_oracle(model, built_library, case):
    from hippopt_b200 import naming

    kw = CASES_A[case]
    if kw is None:
        ev, nlp = pose(model, **distinct_cost_settings("pose"))
    else:
        ev, nlp = kino(model, **kw, **distinct_cost_settings("kino"))
    x, p, lam, _ = inputs(ev, model, 3, seed=301)
    compare(ev, nlp, x, p, lam, SIGMA3.copy(), longdouble=kw is not None and kw.get("smooth", False), label=case)
    if kw is None:
        return
    # the named cost values (hb_eval_cost_terms) carry the same weights
    X, P = (torch.tensor(a, device=dev()) for a in (x, p))
    terms = ev.cost_terms(X, P).cpu().numpy()
    ref = nlp.eval_cost_terms(x, p)
    slots = naming.cost_slots(ev.layout)
    assert set(slots) == set(nlp.cost_names)
    scale = np.abs(ref).max(axis=1)
    for j, name in enumerate(nlp.cost_names):
        k, s = slots[name]
        d = np.abs(terms[:, k, s] - ref[:, j])
        ok = (d <= RTOL * np.abs(ref[:, j])) | (d <= 2.3e-16 * scale)
        assert ok.all(), f"{name}: {terms[:, k, s]} vs {ref[:, j]}"


# ------------------------------------------------------------------------------------------------ b. one term at a time
TERM_CASES = [("kino", n) for n in KINO_MULTIPLIERS] + [("pose", n) for n in POSE_MULTIPLIERS]
TERM_PROBLEM = dict(N=3, fin=True, per=True)


def term_problem(model, kind, name):
    s = only_term(kind, name) if name != "all" else distinct_cost_settings(kind)
    return kino(model, **TERM_PROBLEM, **s) if kind == "kino" else pose(model, **s)


@pytest.fixture(scope="module")
def term_inputs(model, built_library):
    """Per problem kind: x, p and random lam_g shared by every settings variant."""
    out = {}
    for kind in ("kino", "pose"):
        ev, _ = term_problem(model, kind, "all")
        x, p, lam, _ = inputs(ev, model, 2, seed=302)
        out[kind] = (x, p, lam)
    return out


@pytest.mark.parametrize("kind,name", TERM_CASES)
def test_one_cost_term_against_oracle(model, term_inputs, kind, name):
    """lam_g = 0: f, grad_f and hess_l are the one term; each compared at 1e-10 of its own size."""
    ev, nlp = term_problem(model, kind, name)
    x, p, lam = term_inputs[kind]
    out, _ = compare(ev, nlp, x, p, np.zeros_like(lam), SIGMA2.copy(), label=f"{kind}:{name}")
    assert np.abs(out["grad_f"]).max() > 0.0 and np.abs(out["hess"]).max() > 0.0  # the term is not empty


@pytest.mark.parametrize("kind", ["kino", "pose"])
def test_all_costs_off(model, term_inputs, kind):
    """Every multiplier 0 and random lam_g: f and grad_f are exactly 0, hess_l is the constraints' Hessian alone."""
    ev, nlp = term_problem(model, kind, None)
    x, p, lam = term_inputs[kind]
    out, _ = compare(ev, nlp, x, p, lam, SIGMA2.copy(), label=f"{kind}: no cost")
    assert np.all(out["f"] == 0.0) and np.all(out["grad_f"] == 0.0)


@pytest.mark.parametrize("kind", ["kino", "pose"])
def test_cost_terms_add_up_and_leave_the_constraints_alone(model, term_inputs, kind):
    """No oracle: the kernels' outputs are linear in the multipliers.  The per-term evaluations (lam_g = 0) plus the
    all-off evaluation (random lam_g) give the all-on evaluation to 1e-12 in the parity metric; g and jac_g are
    bit-identical across every settings variant."""
    from oracle import parity

    x, p, lam = term_inputs[kind]
    sigma = SIGMA2.copy()
    ev, _ = term_problem(model, kind, "all")
    whole = run(ev, x, p, lam, sigma)
    acc = run(term_problem(model, kind, None)[0], x, p, lam, sigma)
    for name in (KINO_MULTIPLIERS if kind == "kino" else POSE_MULTIPLIERS):
        part = run(term_problem(model, kind, name)[0], x, p, np.zeros_like(lam), sigma)
        for k in ("g", "jac"):
            assert np.array_equal(part[k], whole[k]), (name, k)
        for k in ("f", "grad_f", "hess"):
            acc[k] = acc[k] + part[k]
    for k in ("g", "jac"):
        assert np.array_equal(acc[k], whole[k]), k
    worst = parity.check_all(acc, whole, ev.jac_sparsity(), ev.hess_sparsity(), x, rtol=1e-12,
                             keys=("f", "grad_f", "hess"))
    print(f"{kind} linearity worst relative errors:", {k: f"{v:.2e}" for k, v in worst.items()})


# ------------------------------------------------------------------------------------------------ c. geometry as data
YAW_TRIPLES = list(itertools.permutations(range(4), 3))
LS_TERMS = ("contacts_centroid_cost_multiplier", "foot_yaw_regularization_cost_multiplier",
            "force_regularization_cost_multiplier")


def least_squares_only():
    """The three least-squares terms of the contact kernel (centroid, foot yaw, force ratio) at distinct weights, every
    other multiplier 0: the yaw rows are checked at the size of the rows that share their closed form."""
    s = distinct_cost_settings("kino")
    for n in KINO_MULTIPLIERS:
        if n not in LS_TERMS:
            s[n] = 0.0
    return s


@pytest.fixture(scope="module")
def yaw_reference(model, built_library):
    """g and jac_g of the default triple, which every other triple must reproduce bit for bit."""
    ev, _ = kino(model, 2, **least_squares_only())
    x, p, lam, sigma = two_instances(ev, model, seed=303)
    return (x, p, lam, sigma), run(ev, x, p, lam, sigma)


@pytest.mark.parametrize("yaw", YAW_TRIPLES, ids=lambda t: "".join(map(str, t)))
def test_yaw_points_against_oracle(model, yaw_reference, yaw):
    (x, p, lam, sigma), ref = yaw_reference
    ev, nlp = kino(model, 2, yaw_points=yaw, **least_squares_only())
    out, _ = compare(ev, nlp, x, p, lam, sigma, label=f"yaw {yaw}")
    assert np.array_equal(out["g"], ref["g"]) and np.array_equal(out["jac"], ref["jac"])


@pytest.fixture(scope="module")
def arm_model():
    from hippopt_b200.robot_model import ERGOCUB_JOINTS, RobotModel, synthetic_ergocub_urdf

    return RobotModel.from_urdf(synthetic_ergocub_urdf(), ERGOCUB_JOINTS, "root_link",
                                frames=["l_sole", "r_sole", "chest", "l_forearm"])


@pytest.mark.parametrize("kind", ["kino", "pose"])
@pytest.mark.parametrize("frame", ["root_link", "l_sole", "l_forearm"])
def test_frame_cost_body_against_oracle(model, arm_model, built_library, kind, frame):
    """The frame-cost body as data: the root (body 0, whose adjoints leave the sweep at the base), a foot body (frame
    cost and contact forces on one body) and an arm leaf.  Once with the frame cost alone, once with every term on;
    g and jac_g do not depend on the frame-cost body."""
    m = arm_model if frame == "l_forearm" else model
    alone = only_term(kind, "desired_frame_quaternion_cost_multiplier")
    every = distinct_cost_settings(kind)
    make = (lambda s, **kw: kino(m, 3, fin=True, **s, **kw)) if kind == "kino" else (lambda s, **kw: pose(m, **s, **kw))
    base_ev, _ = make(alone)
    x, p, lam, sigma = two_instances(base_ev, m, seed=304)
    chest = run(base_ev, x, p, lam, sigma)
    for s in (alone, every):
        ev, nlp = make(s, frame_quaternion_cost_frame=frame)
        out, _ = compare(ev, nlp, x, p, lam, sigma, label=f"{kind} frame {frame}{' alone' if s is alone else ''}")
        assert np.array_equal(out["g"], chest["g"]) and np.array_equal(out["jac"], chest["jac"])
        if s is alone:
            assert not np.array_equal(out["grad_f"], chest["grad_f"])  # another body: another cost


@pytest.mark.parametrize("kind", ["kino", "pose"])
def test_swapped_feet_against_oracle(model, built_library, kind):
    feet = ("r_sole", "l_sole")
    s = distinct_cost_settings(kind)
    ev, nlp = kino(model, 3, fin=True, foot_frames=feet, **s) if kind == "kino" else pose(model, foot_frames=feet, **s)
    x, p, lam, sigma = two_instances(ev, model, seed=305)
    compare(ev, nlp, x, p, lam, sigma, label=f"{kind} swapped feet")


# ------------------------------------------------------------------------------------------------ d. zero weights
def test_config4_without_centroid_cost(model, built_library):
    """The reference's periodic-step configuration sets contacts_centroid_cost_multiplier = 0
    (main_periodic_step.py:94): its structure (final state and periodicity) at N = 4, every other weight default."""
    ev, nlp = kino(model, 4, fin=True, per=True, contacts_centroid_cost_multiplier=0.0)
    x, p, lam, _ = inputs(ev, model, 3, seed=306)
    compare(ev, nlp, x, p, lam, SIGMA3.copy(), label="config 4, no centroid cost")


def test_zero_com_velocity_weights(model, built_library):
    """com_linear_velocity_cost_weights = (0, 0, 0): the oracle simplifies 0 * expr away and has fewer Hessian
    entries than the layout; the kernel's values there must be exactly 0."""
    ev, nlp = kino(model, 3, com_linear_velocity_cost_weights=(0.0, 0.0, 0.0))
    assert nlp.hess_structure()[1].size < ev.nnz_h
    x, p, lam, _ = inputs(ev, model, 3, seed=307)
    compare(ev, nlp, x, p, lam, SIGMA3.copy(), label="zero CoM-velocity weights")
