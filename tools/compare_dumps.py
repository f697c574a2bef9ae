"""Compare two `bench.py --dump-outputs` directories with the parity metric of the tests (oracle/parity.py).

    python tools/compare_dumps.py BASE_DIR NEW_DIR [--rtol 1e-12]

BASE_DIR is taken as the reference.  Both runs must come from the same bench arguments (the inputs depend only on
them), so that the two directories hold the same instances.  Prints the worst relative error of f, grad_f, g, jac and
hess, and the share of entries that are bit-identical; exits with 1 when an error exceeds --rtol.

The dumps do not hold x, so g is measured with the x scale of oracle/parity.py::check_g set to 1: a stricter floor than
the parity tests use (they take max(1, ||x||_inf))."""
from __future__ import annotations

import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

NAMES = ("f", "grad_f", "g", "jac", "hess")


def compare(base_dir: str, new_dir: str, horizon: int) -> dict:
    """{name: (worst relative error, share of bit-identical entries)} of new_dir against base_dir."""
    from hippopt_b200.kino_layout import KinoLayout, KinoSettings
    from hippopt_b200.robot_model import synthetic_ergocub
    from oracle import parity

    base = {n: np.load(os.path.join(base_dir, f"{n}.npy")) for n in NAMES}
    new = {n: np.load(os.path.join(new_dir, f"{n}.npy")) for n in NAMES}
    for n in NAMES:
        if base[n].shape != new[n].shape:
            raise ValueError(f"{n}: shapes differ, {base[n].shape} against {new[n].shape}")
    lay = KinoLayout(synthetic_ergocub(), KinoSettings(horizon=horizon))
    if base["jac"].shape[1] != len(lay.jac_row) or base["hess"].shape[1] != len(lay.hess_row):
        raise ValueError(f"the dumps do not have the sparsity of horizon {horizon}")
    x = np.zeros((base["g"].shape[0], 1))
    worst = parity.check_all(new, base, (lay.jac_colind, lay.jac_row), (lay.hess_colind, lay.hess_row), x,
                             rtol=np.inf)
    return {n: (worst[n], float(np.mean(base[n] == new[n]))) for n in NAMES}


def main(argv=None) -> int:
    import bench

    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("base_dir")
    ap.add_argument("new_dir")
    ap.add_argument("--rtol", type=float, default=1e-12)
    ap.add_argument("--horizon", type=int, default=bench.HORIZON)
    args = ap.parse_args(argv)
    res = compare(args.base_dir, args.new_dir, args.horizon)
    ok = True
    for n, (err, same) in res.items():
        flag = "ok" if err <= args.rtol else "FAIL"
        ok &= err <= args.rtol
        print(f"{n:7s} worst relative error {err:.3e}  bit-identical {100 * same:6.2f} %  {flag}")
    print(f"{'all within' if ok else 'NOT within'} rtol {args.rtol:.1e}")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
