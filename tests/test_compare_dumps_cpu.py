"""tools/compare_dumps.py on synthetic dump directories: identical dumps pass, a perturbation above --rtol fails."""
import importlib.util
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tool():
    spec = importlib.util.spec_from_file_location("compare_dumps", os.path.join(ROOT, "tools", "compare_dumps.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _write(d, arrays):
    os.makedirs(d, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(d, f"{n}.npy"), a)


def test_compare_dumps_passes_equal_and_flags_a_perturbation(tmp_path, capsys):
    import bench
    from hippopt_b200.kino_layout import KinoLayout, KinoSettings
    from hippopt_b200.robot_model import synthetic_ergocub

    lay = KinoLayout(synthetic_ergocub(), KinoSettings(horizon=bench.HORIZON))
    rng = np.random.default_rng(3)
    B = 2
    base = {"f": rng.standard_normal(B), "grad_f": rng.standard_normal((B, lay.n_x)), "g": rng.standard_normal((B, lay.m)),
            "jac": rng.standard_normal((B, len(lay.jac_row))), "hess": rng.standard_normal((B, len(lay.hess_row)))}
    _write(tmp_path / "base", base)
    _write(tmp_path / "same", base)
    tool = _tool()
    assert tool.main([str(tmp_path / "base"), str(tmp_path / "same")]) == 0
    res = tool.compare(str(tmp_path / "base"), str(tmp_path / "same"), bench.HORIZON)
    assert all(err == 0.0 and same == 1.0 for err, same in res.values())

    moved = {n: a.copy() for n, a in base.items()}
    i = int(np.argmax(np.abs(moved["hess"][1])))
    moved["hess"][1, i] *= 1.0 + 1e-9
    _write(tmp_path / "moved", moved)
    assert tool.main([str(tmp_path / "base"), str(tmp_path / "moved")]) == 1
    assert "hess    worst relative error 1.0" in capsys.readouterr().out
