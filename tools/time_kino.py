"""Developer timing: kinodynamic evaluator at config-3 size (or, with "stairs", the config-5 problem: smooth-step
terrain, horizon 50, 512 instances; with "tilted", the same problem on kernel terrain 2: the stairs written as two
tilted_steps records, so that the two contact kernels evaluate the same terrain), per-kernel CUDA-event times for the
masks a solver uses."""
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
from hippopt_b200.evaluator import ALL, KinoEvaluator  # noqa: E402
from hippopt_b200.kino_layout import KinoSettings  # noqa: E402
from hippopt_b200.robot_model import synthetic_ergocub  # noqa: E402
from hippopt_b200.workloads import kino_batch  # noqa: E402

model = synthetic_ergocub()
stairs = "stairs" in sys.argv
tilted = "tilted" in sys.argv
nums = [int(a) for a in sys.argv[1:] if a.isdigit()]
if stairs:
    st, B = KinoSettings(horizon=50, terrain="smooth_steps", n_terrain_params=10, final_state_constraint=True), 512
elif tilted:
    st, B = KinoSettings(horizon=50, terrain="tilted_steps", n_terrain_params=20, final_state_constraint=True), 512
else:
    st, B = KinoSettings(horizon=30), 1024
B = nums[0] if nums else B
ev = KinoEvaluator(model, st)
N = ev.layout.N
if tilted:  # the stairs of the "stairs" mode, (l, w, height, ox, oy) x 2 -> two flat steps at z = 0, yaw 0
    from hippopt_b200.kino_layout import KinoLayout

    stairs_lay = KinoLayout(model, KinoSettings(horizon=50, terrain="smooth_steps", n_terrain_params=10,
                                                final_state_constraint=True))
    x, p10, lam, sigma = kino_batch(stairs_lay, model, B, seed=2)
    o = stairs_lay.po.terrain
    p = np.zeros((B, ev.layout.n_p))
    p[:, :o] = p10[:, :o]
    for s in range(2):
        p[:, o + 10 * s:o + 10 * s + 5] = p10[:, o + 5 * s:o + 5 * s + 5]
        p[:, o + 10 * s + 9] = 1.0
else:
    x, p, lam, sigma = kino_batch(ev.layout, model, B, seed=2)
d = torch.device("cuda:0")
X, P, L, S = (torch.tensor(a, device=d) for a in (x, p, lam, sigma))
for mask, name in ((ALL, "f+g+grad+jac+hess"), (ALL & ~16, "f+g+grad+jac"), (16, "hess"), (1 | 4, "f+g")):
    for _ in range(5):
        ev.eval(mask, X, P, L, S)
    torch.cuda.synchronize()
    ev.profile(True)
    t0 = time.perf_counter()
    reps = 30
    for _ in range(reps):
        ev.eval(mask, X, P, L, S)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / reps
    ms, n = ev.profile_read()
    ev.profile(False)
    print(f"{name:20s} {dt * 1e3:7.3f} ms  {B * N / dt:.3e} knot-evals/s   " +
          " ".join(f"{k}={v / n:.3f}" for k, v in ms.items()))
