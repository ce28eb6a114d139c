"""The C-ABI library loads on a box without a GPU and exports every symbol include/wrsn_b200.h declares
(no compute calls here); layouts are consistent; the host layer refuses to run without a device."""
import ctypes
import os
import re

import pytest

from multi_agent_rl_wrsn_b200 import _lib
from tests.helpers import REPO


def _declared_functions():
    with open(os.path.join(REPO, "include", "wrsn_b200.h")) as f:
        src = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return sorted(set(re.findall(r"\b(wrsn_\w+)\s*\(", src)))


@pytest.fixture(scope="module")
def cuda_so():
    import __graft_entry__ as g
    g.build()
    return ctypes.CDLL(_lib.LIB_PATH)


def test_exports_every_declared_symbol(cuda_so):
    names = _declared_functions()
    assert len(names) >= 17
    for n in names:
        assert hasattr(cuda_so, n), n


def test_emulation_exports_the_same_abi():
    emu = ctypes.CDLL(os.path.join(REPO, "tests", "emu", "libwrsn_emu.so"))
    for n in _declared_functions():
        assert hasattr(emu, n), n


def test_layout_and_enums(cuda_so):
    L = _lib._bind(cuda_so)
    e = _lib.enums()
    d = _lib.Dims()
    d.B, d.N, d.T, d.M, d.S, d.Emax, d.TEmax, d.n_scen = 4096, 100, 100, 3, 100, 240, 130, 4
    assert L.wrsn_dims_finalize(ctypes.byref(d)) == 0
    assert d.Npad == 112 and d.W == 4 and d.Tw == 4 and d.threads == 32
    off = (ctypes.c_int64 * e["WRSN_F_COUNT"])()
    assert L.wrsn_state_layout(ctypes.byref(d), off) == 0
    offs = list(off)
    assert offs == sorted(offs) and all(o % 16 == 0 for o in offs)
    assert offs[e["WRSN_F_LOGTICK"]] == d.state_resident_bytes and d.state_bytes > d.state_resident_bytes
    assert d.smem_bytes <= 227 * 1024
    soff = (ctypes.c_int64 * e["WRSN_S_COUNT"])()
    assert L.wrsn_scen_layout(ctypes.byref(d), soff) == 0
    assert list(soff) == sorted(soff)
    bad = _lib.Dims()
    bad.B, bad.N, bad.T, bad.M, bad.S = 1, 100, 100, 99, 100
    assert L.wrsn_dims_finalize(ctypes.byref(bad)) == 0
    assert L.wrsn_state_layout(ctypes.byref(bad), off) != 0            # M > WRSN_MAX_MC is rejected
    assert b"bad dims" in L.wrsn_last_error()


def test_emulation_dims_and_layouts_equal_the_cuda_library(cuda_so):
    """Both libraries compile the same host side of the ABI: the same dims, thread counts and layouts, the same rejections."""
    libs = [_lib._bind(cuda_so), _lib._bind(ctypes.CDLL(os.path.join(REPO, "tests", "emu", "libwrsn_emu.so")))]
    e = _lib.enums()

    def finalize(L, N, T, M, S, rounds=0):
        d = _lib.Dims()
        d.B, d.N, d.T, d.M, d.S, d.Emax, d.TEmax, d.n_scen = 8, N, T, M, S, 6 * N, 2 * T, 2
        rc = L.wrsn_dims_finalize(ctypes.byref(d))
        d.step_budget, d.step_rounds = 60, rounds
        off = (ctypes.c_int64 * e["WRSN_F_COUNT"])()
        soff = (ctypes.c_int64 * e["WRSN_S_COUNT"])()
        rcs = (rc, L.wrsn_state_layout(ctypes.byref(d), off), L.wrsn_scen_layout(ctypes.byref(d), soff))
        return rcs, {f: getattr(d, f) for f, _ in d._fields_}, list(off), list(soff)

    for N in (50, 100, 150, 500, 1000):
        for T, M, S in ((N, 3, 100), (2 * N, 10, 64), (7, 1, 37)):
            got = [finalize(L, N, T, M, S) for L in libs]
            assert got[0] == got[1], (N, T, M, S)
            assert got[0][0] == (0, 0, 0)
    assert [finalize(L, 150, 150, 3, 100)[1]["threads"] for L in libs] == [64, 64]
    for kw, msg in ((dict(M=e["WRSN_MAX_MC"] + 1), b"bad dims"), (dict(M=3, rounds=-1), b"step_rounds")):
        for L in libs:
            rcs = finalize(L, N=100, T=100, S=100, **kw)[0]
            assert rcs[1] != 0 and rcs[2] != 0 and msg in L.wrsn_last_error()


def test_emulation_entry_point_checks_equal_the_cuda_library(cuda_so):
    """wrsn_observe, wrsn_k_charge and both decode entry points check their arguments in the shared host side of the ABI: both
    libraries refuse the same inputs with the same message.  No input here passes the checks, so nothing is launched."""
    import numpy as np
    libs = [_lib._bind(cuda_so), _lib._bind(ctypes.CDLL(os.path.join(REPO, "tests", "emu", "libwrsn_emu.so")))]
    max_mc = _lib.enums()["WRSN_MAX_MC"]

    def dims(L, M=3, S=100, finalize=True):
        d = _lib.Dims()
        d.B, d.N, d.T, d.M, d.S, d.Emax, d.TEmax, d.n_scen = 2, 100, 100, M, S, 600, 200, 1
        if finalize:
            assert L.wrsn_dims_finalize(ctypes.byref(d)) == 0
        return d

    # zeroed buffers large enough for every case, and no row with an observer: an entry point that skipped its checks would
    # return 0 instead of touching memory it does not own
    big = dims(libs[0], M=max_mc + 1, S=177)
    B, N, M, S = big.B, big.N, big.M, big.S
    arrays = dict(scen=np.zeros(big.scen_bytes * big.n_scen, np.uint8), scen_id=np.zeros(B, np.int32),
                  state=np.zeros(big.state_bytes * B, np.uint8), agent=np.full(B, -1, np.int32),
                  obs=np.zeros(B * 4 * S * S, np.float64), map=np.zeros(B * S * S, np.float64),
                  action=np.zeros(B * 3, np.float64), node=np.zeros(B * N, np.float64), mc=np.zeros(B * M, np.float64))
    weights = (ctypes.c_float * 9)(*([1.0] * 9))

    def call(L, name, d, null=None, channels=4):
        p = {k: (None if k == null else a.ctypes.data) for k, a in arrays.items()}
        rd = ctypes.byref(d)
        if name == "observe":
            rc = L.wrsn_observe(rd, p["scen"], p["scen_id"], p["state"], p["agent"], p["obs"], 1, None)
        elif name == "k_charge":
            rc = L.wrsn_k_charge(rd, p["scen"], p["scen_id"], p["state"], None, p["node"], p["mc"], None)
        elif name == "decode_density_map":
            rc = L.wrsn_decode_density_map(rd, p["scen"], p["scen_id"], p["state"], p["agent"], p["map"], 1, p["action"], None)
        else:
            rc = L.wrsn_decode_linear_controller(rd, p["scen"], p["scen_id"], p["state"], p["agent"], p["obs"], channels, weights,
                                                 p["action"], None)
        return rc, L.wrsn_last_error()

    every = ("observe", "k_charge", "decode_density_map", "decode_linear_controller")
    cases = [(every, dict(finalize=False), {}, b"dims not finalized"),
             (every, dict(M=max_mc + 1), {}, b"bad dims"),
             (every, {}, dict(null="state"), b"NULL argument"),
             (every, {}, dict(null="scen_id"), b"NULL argument"),
             (("observe",), {}, dict(null="obs"), b"NULL argument"),
             (("k_charge",), {}, dict(null="node"), b"NULL argument"),
             (("decode_density_map",), {}, dict(null="map"), b"NULL argument"),
             (("decode_linear_controller",), {}, dict(channels=0), b"1 to 8 channels"),
             (("decode_linear_controller",), {}, dict(channels=9), b"1 to 8 channels"),
             (("decode_density_map", "decode_linear_controller"), dict(S=177), {}, b"map_size = 177")]
    for names, dkw, ckw, msg in cases:
        for name in names:
            got = [call(L, name, dims(L, **dkw), **ckw) for L in libs]
            assert got[0] == got[1], (name, dkw, ckw, got)
            assert got[0][0] == -1 and msg in got[0][1], (name, dkw, ckw, got)


def test_no_cpu_path():
    """Without a GPU the product host layer must refuse loudly, not fall back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from multi_agent_rl_wrsn_b200 import BatchedWRSN, synthetic
    from tests import helpers
    helpers.use_cuda_build_lazy()
    with pytest.raises(RuntimeError):
        BatchedWRSN(synthetic(num_nodes=20, num_targets=20, seed=0), num_agent=1, num_envs=1)
    with pytest.raises(RuntimeError):
        BatchedWRSN(synthetic(num_nodes=20, num_targets=20, seed=0), num_agent=1, num_envs=1, device="cpu")
