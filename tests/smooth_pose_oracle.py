"""The pose finder's oracle on the stairs: `oracle.pose_finder.build` on the two smooth steps, with their ten
parameters (l, w, height, ox, oy) x 2 appended to p as runtime data (p = 212), as `oracle.kinodynamic` does for the
kinodynamic OCP.

`pose_finder.build` binds the terrain rows (complementarity, height, normal, friction) to their point's x and the
scalar parameters only; here it builds them over symbolic terrain parameters and each of the four templates is then
re-bound with the parameter symbols as extra inputs, pointing at the appended slots of p.  Rows, costs, names and
their order are exactly those of `pose_finder.build`."""
import dataclasses

import numpy as np

from oracle import expressions as ex
from oracle import pose_finder as pf
from oracle import sx
from oracle.nlp import Template

TERRAIN_ROWS = ("complementarity", "height", "normal", "friction")
N_TERRAIN = ex.TwoSmoothSteps.N_PARAMS


def build(model, st: pf.Settings | None = None):
    """(nlp, layout) of the pose finder on the smooth steps; p = [the 202 planar parameters, terrain (10)]."""
    tp = sx.syms("tp", N_TERRAIN)
    st = dataclasses.replace(st or pf.Settings(), terrain=ex.TwoSmoothSteps().with_params(tp))
    nlp, lay = pf.build(model, st)
    lay.terrain = nlp.n_x + nlp.n_p
    tp_idx = np.arange(lay.terrain, lay.terrain + N_TERRAIN)
    nlp.n_p += N_TERRAIN
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
