"""ctypes binding of ``libwrsn_b200.so`` (C ABI: ``include/wrsn_b200.h``).

There is no CPU path: if the CUDA library has not been built (``python -c "import __graft_entry__ as g;
g.build()"``) or no sm_100 device is visible, constructing a simulator raises.
"""
import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(_HERE)
LIB_PATH = os.path.join(_HERE, "csrc", "libwrsn_b200.so")
HEADER = os.path.join(_REPO, "include", "wrsn_b200.h")

_lib = None
_enums = None


class Dims(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "B", "N", "T", "M", "S", "Emax", "TEmax", "n_scen", "threads",
        "Npad", "W", "Tw", "n_slot", "state_bytes", "state_resident_bytes", "scen_bytes", "smem_bytes", "obs_pitch",
        "step_budget")] + [("obs_sigma_cells", C.c_float), ("step_rounds", C.c_int32)]


class Request(C.Structure):
    _fields_ = [("agent_id", C.c_void_p), ("terminal", C.c_void_p), ("reward", C.c_void_p), ("now", C.c_void_p),
                ("action", C.c_void_p), ("detail", C.c_void_p), ("flags", C.c_void_p), ("stats", C.c_void_p), ("sticky", C.c_void_p), ("order", C.c_void_p)]


def enums():
    """The WRSN_* enum values, parsed from the header so Python and C can never disagree."""
    global _enums
    if _enums is not None:
        return _enums
    with open(HEADER) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    out = {}
    for m in re.finditer(r"#define\s+(WRSN_\w+)\s+(\d+)", src):
        out[m.group(1)] = int(m.group(2))
    for body in re.findall(r"enum\s*\{(.*?)\}", src, flags=re.S):
        val = -1
        for item in body.split(","):
            item = item.strip()
            if not item:
                continue
            if "=" in item:
                name, expr = [s.strip() for s in item.split("=", 1)]
                val = int(eval(expr, {}, out))          # noqa: S307 - header arithmetic over earlier enumerators
            else:
                name = item
                val += 1
            out[name] = val
    _enums = out
    return out


def _bind(L):
    vp, ip = C.c_void_p, C.c_int
    dp = C.POINTER(Dims)
    L.wrsn_last_error.restype = C.c_char_p
    L.wrsn_abi_version.restype = ip
    L.wrsn_field_count.argtypes = [ip]
    L.wrsn_dims_finalize.argtypes = [dp]
    L.wrsn_state_layout.argtypes = [dp, C.POINTER(C.c_int64)]
    L.wrsn_scen_layout.argtypes = [dp, C.POINTER(C.c_int64)]
    L.wrsn_device_ok.restype = ip
    L.wrsn_build_obs_tables.argtypes = [dp, vp, vp]
    L.wrsn_init_network.argtypes = [dp, vp, vp, vp, vp, ip, vp]
    L.wrsn_run_until.argtypes = [dp, vp, vp, vp, vp, vp, vp]
    L.wrsn_reset_finish.argtypes = [dp, vp, vp, vp, vp, C.POINTER(Request), vp]
    L.wrsn_reset_from_snapshot.argtypes = [dp, vp, vp, vp, vp, vp, C.POINTER(Request), vp]
    L.wrsn_step.argtypes = [dp, vp, vp, vp, vp, vp, vp, C.POINTER(Request), vp]
    L.wrsn_rollout_step.argtypes = [dp, vp, vp, vp, vp, vp, C.POINTER(Request), vp, ip, vp]
    L.wrsn_observe.argtypes = [dp, vp, vp, vp, vp, vp, ip, vp]
    L.wrsn_record_transitions.argtypes = [dp, C.POINTER(Request), C.c_int64, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.wrsn_copy_rows.argtypes = [dp, C.c_int32, vp, C.POINTER(Request), vp, vp, C.c_int32, vp, C.POINTER(Request), vp, vp,
                                 C.c_int32, vp]
    L.wrsn_fitness.argtypes = [dp, vp, vp, vp, vp, vp, vp]
    L.wrsn_k_charge.argtypes = [dp, vp, vp, vp, vp, vp, vp, vp]
    L.wrsn_decode_density_map.argtypes = [dp, vp, vp, vp, vp, vp, ip, vp, vp]
    L.wrsn_decode_linear_controller.argtypes = [dp, vp, vp, vp, vp, vp, ip, C.POINTER(C.c_float), vp, vp]
    L.wrsn_heuristic_action.argtypes = [dp, vp, vp, vp, vp, ip, vp, vp]
    L.wrsn_heuristic_candidates.argtypes = [dp, vp, vp, vp, vp, ip, ip, vp, vp, vp]
    L.wrsn_rule_rollout.argtypes = [dp, vp, vp, vp, vp, ip, vp, C.c_int64, C.c_int32, vp, vp, C.POINTER(Request), vp]
    for k in ("wrsn_k_bfs", "wrsn_k_drain", "wrsn_k_bookkeep", "wrsn_k_reward"):
        getattr(L, k).argtypes = [dp, vp, vp, vp, vp]
    e = enums()
    if L.wrsn_abi_version() != e["WRSN_ABI_VERSION"]:
        raise RuntimeError("libwrsn_b200.so ABI %d != header %d: rebuild" % (L.wrsn_abi_version(), e["WRSN_ABI_VERSION"]))
    for which, key in enumerate(("WRSN_P_LEN", "WRSN_H_LEN", "WRSN_MC_LEN", "WRSN_PR_LEN", "WRSN_F_COUNT", "WRSN_S_COUNT")):
        if L.wrsn_field_count(which) != e[key]:
            raise RuntimeError("libwrsn_b200.so disagrees with include/wrsn_b200.h on %s: rebuild" % key)
    return L


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("CUDA extension %s is missing - build it first (python -c 'import __graft_entry__ as g; "
                               "g.build()').  This package has no CPU fallback." % LIB_PATH)
        _lib = _bind(C.CDLL(LIB_PATH))
    return _lib


def check(rc, L):
    if rc != 0:
        raise RuntimeError("wrsn_b200: " + L.wrsn_last_error().decode())
