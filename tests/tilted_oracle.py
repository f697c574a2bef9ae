"""Oracle of the general smooth-step terrain (``terrain="tilted_steps"``, kernel terrain 2): `SmoothTerrain.step` with
yaw, origin height and the tilted top (SURVEY.md A.10, smooth_terrain.py:235-264), K steps summed as a TerrainSum over
runtime parameters (l, w, height, ox, oy, oz, yaw, n_x, n_y, n_z) per step, and the kinodynamic and pose-finder
oracles built on it.

    (x_t, y_t) = R_z(yaw)^T (p - o)_{xy},  g = (2 x_t / l)^10 + (2 y_t / w)^10,
    z_t = exp(-g^20) pi(x_t, y_t),  pi = height - n_x / n_z x_t - n_y / n_z y_t,  h = p_z - z_t - o_z
"""
import dataclasses

import numpy as np

from oracle import expressions as ex
from oracle import kinodynamic as kd
from oracle import pose_finder as pf
from oracle import sx
from oracle.nlp import Template

N_STEP = 10  # parameters per step


class TiltedStep(ex.SmoothStep):
    """`ex.SmoothStep` with the tilted top of smooth_terrain.py:255-263: the box's top is the plane through
    (0, 0, height) in step coordinates with the normal (n_x, n_y, n_z); (0, 0, 1) is the flat top."""

    def __init__(self, length, width, height, origin=(0.0, 0.0, 0.0), yaw=0.0, normal=(0.0, 0.0, 1.0)):
        super().__init__(length, width, height, origin=origin, yaw=yaw)
        self.n = normal

    def height(self, p):
        dx = p[0] - self.origin[0]
        dy = p[1] - self.origin[1]
        c, s = sx.cos(self.yaw), sx.sin(self.yaw)
        xt = c * dx + s * dy
        yt = c * dy - s * dx
        g = sx.powc(2.0 * xt / self.length, 2.0 * self.e) + sx.powc(2.0 * yt / self.width, 2.0 * self.e)
        top = self.h - self.n[0] / self.n[2] * xt - self.n[1] / self.n[2] * yt
        zt = sx.exp(-sx.powc(g, 2.0 * self.s)) * top
        return p[2] - (zt + self.origin[2])


class TiltedSteps(ex.Terrain):
    """K tilted steps as ((step_0 + step_1) + step_2) + ..., TerrainSum by TerrainSum, over 10 K runtime parameters."""

    def __init__(self, K: int, params=None):
        self.K, self.params = K, params
        self.N_PARAMS = N_STEP * K

    def with_params(self, tp):
        assert len(tp) == self.N_PARAMS
        return TiltedSteps(self.K, tp)

    def steps(self):
        tp = self.params
        return [TiltedStep(tp[10 * s], tp[10 * s + 1], tp[10 * s + 2], origin=tuple(tp[10 * s + 3:10 * s + 6]),
                           yaw=tp[10 * s + 6], normal=tuple(tp[10 * s + 7:10 * s + 10])) for s in range(self.K)]

    def height(self, p):
        steps = self.steps()
        t = steps[0]
        for s in steps[1:]:
            t = ex.TerrainSum(t, s)
        return t.height(p)


def kino_build(model, K: int, **settings):
    """(nlp, layout) of the kinodynamic OCP on K tilted steps: p = [..., terrain (10 K)]."""
    return kd.build(model, kd.Settings(terrain=TiltedSteps(K), terrain_params=N_STEP * K, **settings))


TERRAIN_ROWS = ("complementarity", "height", "normal", "friction")


def pose_build(model, K: int, st: pf.Settings | None = None):
    """(nlp, layout) of the pose finder on K tilted steps, p = [the 202 planar parameters, terrain (10 K)]: the terrain
    rows of `pose_finder.build` re-bound to the appended parameter slots, as tests/smooth_pose_oracle.py does for the
    stairs."""
    n = N_STEP * K
    tp = sx.syms("tp", n)
    st = dataclasses.replace(st or pf.Settings(), terrain=TiltedSteps(K).with_params(tp))
    nlp, lay = pf.build(model, st)
    lay.terrain = nlp.n_x + nlp.n_p
    tp_idx = np.arange(lay.terrain, lay.terrain + n)
    nlp.n_p += n
    lay.n_p = nlp.n_p
    rebound = {}
    apps = []
    for t, binding, off in nlp.row_apps:
        if t.name in TERRAIN_ROWS:
            if id(t) not in rebound:
                rebound[id(t)] = Template(t.name, t.inputs + list(tp), t.rows, lb=t.lb, ub=t.ub)
            t, binding = rebound[id(t)], np.concatenate([binding, tp_idx])
        apps.append((t, binding, off))
    assert len(rebound) == len(TERRAIN_ROWS)
    nlp.row_apps = apps
    return nlp, lay


def stairs_as_tilted(tp10: np.ndarray) -> np.ndarray:
    """(B, 10) stairs parameters (l, w, height, ox, oy) x 2 -> the same terrain as (B, 20) tilted_steps parameters."""
    tp10 = np.atleast_2d(tp10)
    out = np.zeros((tp10.shape[0], 20))
    for s in range(2):
        out[:, 10 * s:10 * s + 5] = tp10[:, 5 * s:5 * s + 5]
        out[:, 10 * s + 9] = 1.0
    return out
