"""ctypes binding of the C ABI declared in include/hippopt_b200.h.

The header is the single source of truth for the configuration-table indices: its enums and
integer ``#define``s are parsed here rather than duplicated.  Loading fails loudly when the CUDA
library has not been built -- there is no CPU fallback (``__graft_entry__.build()`` builds it).
"""
from __future__ import annotations

import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
HEADER = os.path.join(os.path.dirname(_HERE), "include", "hippopt_b200.h")
LIB_PATH = os.environ.get("HIPPOPT_B200_LIB", os.path.join(_HERE, "libhippopt_b200.so"))  # override: kernel tuning


def parse_header(path: str = HEADER) -> dict[str, int]:
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    text = re.sub(r"//[^\n]*", "", text)
    env: dict[str, int] = {}
    # process #defines and enums in file order (later ones reference earlier ones)
    pattern = re.compile(r"#define\s+(\w+)\s+([^\n]+)|enum\s*\{([^}]*)\}", re.S)
    for mt in pattern.finditer(text):
        if mt.group(1):
            name, expr = mt.group(1), mt.group(2).strip()
            if not expr or name.endswith("_H"):
                continue
            try:
                env[name] = int(eval(expr, {"__builtins__": {}}, env))
            except Exception:
                pass
        else:
            nxt = 0
            for item in mt.group(3).split(","):
                item = item.strip()
                if not item:
                    continue
                if "=" in item:
                    name, expr = (s.strip() for s in item.split("=", 1))
                    nxt = int(eval(expr, {"__builtins__": {}}, env))
                else:
                    name = item
                env[name] = nxt
                nxt += 1
    return env


H = parse_header()


class LibraryNotBuilt(RuntimeError):
    pass


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise LibraryNotBuilt(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). hippopt_b200 has no CPU fallback."
        )
    L = ctypes.CDLL(LIB_PATH)
    vp, i32p, i16p, f64p, i64p = (ctypes.c_void_p, ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int16),
                                  ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int64))
    i64 = ctypes.c_int64
    L.hb_kino_create.restype = ctypes.c_int
    L.hb_kino_create.argtypes = [i32p, f64p, i32p, i32p, i16p, i32p, i32p, i32p, ctypes.POINTER(vp)]
    L.hb_toy_create.restype = ctypes.c_int
    L.hb_toy_create.argtypes = [ctypes.c_int32, ctypes.c_int32, ctypes.c_double, ctypes.POINTER(vp)]
    L.hb_destroy.restype = ctypes.c_int
    L.hb_destroy.argtypes = [vp]
    L.hb_dims.restype = ctypes.c_int
    L.hb_dims.argtypes = [vp, i64p, i64p, i64p, i64p, i64p]
    L.hb_pattern_jac.restype = ctypes.c_int
    L.hb_pattern_jac.argtypes = [vp, i64p, i64p]
    L.hb_pattern_hess.restype = ctypes.c_int
    L.hb_pattern_hess.argtypes = [vp, i64p, i64p]
    L.hb_eval.restype = ctypes.c_int
    L.hb_eval.argtypes = [vp, ctypes.c_uint32, vp, vp, ctypes.c_int64, vp, vp, vp, vp, vp, vp, vp, ctypes.c_int64, vp]
    L.hb_kino_attach_tables.restype = ctypes.c_int
    L.hb_kino_attach_tables.argtypes = [vp, i64p, i64p, i64p, i64p, i32p, f64p, i32p, f64p]
    L.hb_bounds.restype = ctypes.c_int
    L.hb_bounds.argtypes = [vp, f64p, f64p, f64p]
    L.hb_save.restype = ctypes.c_int
    L.hb_save.argtypes = [vp, ctypes.c_char_p]
    L.hb_load.restype = ctypes.c_int
    L.hb_load.argtypes = [ctypes.c_char_p, ctypes.POINTER(vp)]
    L.hb_ccs_group_mul.restype = ctypes.c_int
    L.hb_ccs_group_mul.argtypes = [vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, i64, vp]
    L.hb_kkt_assemble_stage.restype = ctypes.c_int
    L.hb_kkt_assemble_stage.argtypes = [i32p, vp, vp, i64, vp, i64, vp, i64, vp, ctypes.c_double, vp, i64, vp, i64, vp, vp,
                                        vp, i64, vp]
    L.hb_external_bind.restype = ctypes.c_int
    L.hb_external_bind.argtypes = [vp]
    L.hb_external_stats.restype = ctypes.c_int
    L.hb_external_stats.argtypes = [i64p, i64p]
    L.hb_eval_cost_terms.restype = ctypes.c_int
    L.hb_eval_cost_terms.argtypes = [vp, vp, vp, ctypes.c_int64, vp, ctypes.c_int64, vp]
    L.hb_debug_sweep_schedule.restype = ctypes.c_int
    L.hb_debug_sweep_schedule.argtypes = [ctypes.c_int32, i32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                          ctypes.c_int32, i32p, i32p]
    L.hb_debug_sweep_schedule_n_base.restype = ctypes.c_int
    L.hb_debug_sweep_schedule_n_base.argtypes = [ctypes.c_int32, i32p, ctypes.c_int32, ctypes.c_int32, ctypes.c_int32,
                                                 ctypes.c_int32, ctypes.c_int32, i32p, i32p]
    L.hb_host_set_parameters.restype = ctypes.c_int
    L.hb_host_set_parameters.argtypes = [vp, vp, ctypes.c_int64, ctypes.c_int64]
    L.hb_eval_host.restype = ctypes.c_int
    L.hb_eval_host.argtypes = [vp, ctypes.c_uint32, vp, vp, vp, vp, vp, vp, vp, vp, ctypes.c_int64]
    L.hb_host_last_traffic.restype = ctypes.c_int
    L.hb_host_last_traffic.argtypes = [vp, i64p, i64p]
    L.hb_host_alloc.restype = ctypes.c_int
    L.hb_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_int64]
    L.hb_host_free.restype = ctypes.c_int
    L.hb_host_free.argtypes = [vp]
    L.hb_lu_factor_batched.restype = ctypes.c_int
    L.hb_lu_factor_batched.argtypes = [vp, vp, vp, ctypes.c_int64, ctypes.c_int64, vp]
    L.hb_lu_solve_batched.restype = ctypes.c_int
    L.hb_lu_solve_batched.argtypes = [vp, vp, vp, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, vp]
    L.hb_debug_lu_plan.restype = ctypes.c_int
    L.hb_debug_lu_plan.argtypes = [ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_int32, i32p]
    L.hb_debug_smooth_terrain.restype = ctypes.c_int
    L.hb_debug_smooth_terrain.argtypes = [vp, vp, ctypes.c_int64, vp, vp]
    L.hb_debug_tilted_terrain.restype = ctypes.c_int
    L.hb_debug_tilted_terrain.argtypes = [vp, ctypes.c_int32, vp, ctypes.c_int64, vp, vp]
    i64 = ctypes.c_int64
    L.hb_interpolate_humanoid_states.restype = ctypes.c_int
    L.hb_interpolate_humanoid_states.argtypes = [i64, i64, i64, vp, vp, vp, vp, i64, i64, vp, i64, i64, vp, vp, i64, i64, vp]
    L.hb_last_launch_count.restype = ctypes.c_int
    L.hb_last_launch_count.argtypes = [vp]
    L.hb_set_option.restype = ctypes.c_int
    L.hb_set_option.argtypes = [vp, ctypes.c_int32, ctypes.c_int32]
    L.hb_last_error.restype = ctypes.c_char_p
    L.hb_last_error.argtypes = []
    L.hb_profile_enable.restype = ctypes.c_int
    L.hb_profile_enable.argtypes = [vp, ctypes.c_int]
    L.hb_profile_read.restype = ctypes.c_int
    L.hb_profile_read.argtypes = [vp, f64p, i64p]
    L.hb_probe_fp64_tflops.restype = ctypes.c_int
    L.hb_probe_fp64_tflops.argtypes = [f64p, vp]
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "hb_kino_create", "hb_toy_create", "hb_destroy", "hb_dims", "hb_pattern_jac", "hb_pattern_hess", "hb_eval",
    "hb_last_launch_count", "hb_last_error", "hb_probe_fp64_tflops", "hb_profile_enable", "hb_profile_read",
    "hb_host_set_parameters", "hb_eval_host", "hb_host_last_traffic", "hb_host_alloc", "hb_host_free",
    "hb_lu_factor_batched", "hb_lu_solve_batched", "hb_debug_lu_plan", "hb_debug_smooth_terrain", "hb_debug_tilted_terrain",
    "hb_set_option", "hb_interpolate_humanoid_states",
    "hb_eval_cost_terms", "hb_debug_sweep_schedule", "hb_debug_sweep_schedule_n_base", "hb_kino_attach_tables",
    "hb_bounds", "hb_save", "hb_load",
    "hb_ccs_group_mul", "hb_external_bind", "hb_external_stats", "hb_kkt_assemble_stage",
] + ['hb_nlp_f', 'hb_nlp_f_n_in', 'hb_nlp_f_n_out', 'hb_nlp_f_sparsity_in', 'hb_nlp_f_sparsity_out', 'hb_nlp_f_work', 'hb_nlp_f_name_in', 'hb_nlp_f_name_out', 'hb_nlp_f_incref', 'hb_nlp_f_decref', 'hb_nlp_f_alloc_mem', 'hb_nlp_f_init_mem', 'hb_nlp_f_free_mem', 'hb_nlp_f_checkout', 'hb_nlp_f_release', 'hb_nlp_g', 'hb_nlp_g_n_in', 'hb_nlp_g_n_out', 'hb_nlp_g_sparsity_in', 'hb_nlp_g_sparsity_out', 'hb_nlp_g_work', 'hb_nlp_g_name_in', 'hb_nlp_g_name_out', 'hb_nlp_g_incref', 'hb_nlp_g_decref', 'hb_nlp_g_alloc_mem', 'hb_nlp_g_init_mem', 'hb_nlp_g_free_mem', 'hb_nlp_g_checkout', 'hb_nlp_g_release', 'hb_nlp_grad_f', 'hb_nlp_grad_f_n_in', 'hb_nlp_grad_f_n_out', 'hb_nlp_grad_f_sparsity_in', 'hb_nlp_grad_f_sparsity_out', 'hb_nlp_grad_f_work', 'hb_nlp_grad_f_name_in', 'hb_nlp_grad_f_name_out', 'hb_nlp_grad_f_incref', 'hb_nlp_grad_f_decref', 'hb_nlp_grad_f_alloc_mem', 'hb_nlp_grad_f_init_mem', 'hb_nlp_grad_f_free_mem', 'hb_nlp_grad_f_checkout', 'hb_nlp_grad_f_release', 'hb_nlp_jac_g', 'hb_nlp_jac_g_n_in', 'hb_nlp_jac_g_n_out', 'hb_nlp_jac_g_sparsity_in', 'hb_nlp_jac_g_sparsity_out', 'hb_nlp_jac_g_work', 'hb_nlp_jac_g_name_in', 'hb_nlp_jac_g_name_out', 'hb_nlp_jac_g_incref', 'hb_nlp_jac_g_decref', 'hb_nlp_jac_g_alloc_mem', 'hb_nlp_jac_g_init_mem', 'hb_nlp_jac_g_free_mem', 'hb_nlp_jac_g_checkout', 'hb_nlp_jac_g_release', 'hb_nlp_hess_l', 'hb_nlp_hess_l_n_in', 'hb_nlp_hess_l_n_out', 'hb_nlp_hess_l_sparsity_in', 'hb_nlp_hess_l_sparsity_out', 'hb_nlp_hess_l_work', 'hb_nlp_hess_l_name_in', 'hb_nlp_hess_l_name_out', 'hb_nlp_hess_l_incref', 'hb_nlp_hess_l_decref', 'hb_nlp_hess_l_alloc_mem', 'hb_nlp_hess_l_init_mem', 'hb_nlp_hess_l_free_mem', 'hb_nlp_hess_l_checkout', 'hb_nlp_hess_l_release']


class EvaluationError(RuntimeError):
    pass


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise EvaluationError(f"{what} failed with code {rc}: {lib().hb_last_error().decode()}")
