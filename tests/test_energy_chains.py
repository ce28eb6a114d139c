"""The exact energy replay at binade edges, against literal fp64 chains.

A node's tick is its own sequence of fp64 subtractions (relays of lower ids, top-up, own packets, relays of higher ids).  Inside
one binade [lo, 2 lo) the engine evaluates it in closed form as a whole number of ulps u: ``sub_chain`` / ``sub_chain_fast``
(every drain tick), the irregular-node table of a whole-cycle batch (``spec_terms``: D1, D2, H and the guards glo / ghi) and the
per-cycle decrement of an uncharged node (``batch_dec``).  A chain that ends exactly on lo is the edge: its last literal
subtraction may fall below lo, where the spacing is u/2, and round to lo - u/2.  Natural trajectories land there with
probability about 1/K (K = 1e8 .. 1e10 ulps per tick), so the cases here are built to land on it.

``tests/emu/energy_probe.cu`` exposes the functions one case at a time; it is compiled here for the host build (g++, the flags of
tests/emu/Makefile) and, under ``-m gpu``, with nvcc and the library's flags, including the whole of wrsn_kernels.cu.  The
reference is a Python loop of ``e -= x`` on Python floats (IEEE doubles); results are compared bit for bit.  Every group of cases
also counts the cases where the closed form with the old lower bound (r >= lo) differs from the literal chain, and fails if there
is none: the cases must reach the edge.

The device-only reward helpers (``wrsn_rcp``, ``wrsn_rsqrt``, ``wrsn_exp_tab``; the host build uses libm) are checked against
mpmath at 50 digits, and the end-to-end cases put crafted energies into the engine and the C oracle and compare the energies bit
for bit after a drain tick, after 40 s of batches and event ticks, and across a second of an active batch."""
import ctypes as C
import math
import os
import shlex
import subprocess

import numpy as np
import pytest
import torch

from tests import helpers
from tests import parity_cases as pc
from tests.helpers import REPO

CSRC = os.path.join(REPO, "multi_agent_rl_wrsn_b200", "csrc")
EMU_DIR = os.path.join(REPO, "tests", "emu")
PROBE_SRC = os.path.join(EMU_DIR, "energy_probe.cu")
PROBE_IN, PROBE_OUT = 10, 8
(OP_SUB_CHAIN, OP_SUB_CHAIN_FAST, OP_SUB_CHAIN_LITERAL, OP_DRAIN_NODE, OP_REPLAY_CYCLES, OP_SPEC_TERMS, OP_BATCH_DEC,
 OP_RCP, OP_RSQRT, OP_EXP_TAB, OP_CHARGE_RUN, OP_MOVE_SPAN) = range(12)
GPU = "cuda:0"
KS = range(9, 15)                                    # binades 2^9 .. 2^14: the scenarios' threshold-to-capacity range
SLACK = 1e-6                                         # the engine's margin above the threshold (replay_cycles, batch_dec)


# ------------------------------------------------------------------ the probe, host and device builds
def _emu_cxxflags():
    with open(os.path.join(EMU_DIR, "Makefile")) as f:
        for line in f:
            if line.startswith("CXXFLAGS"):
                return shlex.split(line.split("=", 1)[1])
    raise AssertionError("CXXFLAGS not found in tests/emu/Makefile")


class Probe:
    def __init__(self, path, device):
        self.L = C.CDLL(path)
        self.L.probe_run.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_int]
        self.L.probe_run.restype = C.c_int
        self.device = device

    def __call__(self, op, rows):
        rows = np.asarray(rows, np.float64)
        if rows.ndim == 1:
            rows = rows[:, None]
        n = rows.shape[0]
        x = np.zeros((n, PROBE_IN))
        x[:, :rows.shape[1]] = rows
        if self.device is None:
            y = np.zeros((n, PROBE_OUT))
            rc = self.L.probe_run(op, x.ctypes.data, y.ctypes.data, n)
        else:
            xt = torch.as_tensor(x, device=self.device)
            yt = torch.zeros((n, PROBE_OUT), dtype=torch.float64, device=self.device)
            rc = self.L.probe_run(op, xt.data_ptr(), yt.data_ptr(), n)
            y = yt.cpu().numpy()
        assert rc == 0 and not y[:, 5].any(), ("probe", op, rc)
        return y


_PROBES = {}


def _probe(kind, tmp_path_factory):
    """the probe for the host build ("cpu") or the device (built once per session and kind)"""
    if kind not in _PROBES:
        out = str(tmp_path_factory.mktemp("energy_probe") / "energy_probe.so")
        inc = ["-I", os.path.join(REPO, "include"), "-I", CSRC]
        if kind == "cpu":
            subprocess.check_call([os.environ.get("CXX", "g++")] + _emu_cxxflags() + inc + ["-x", "c++", "-o", out, PROBE_SRC])
            _PROBES[kind] = Probe(out, None)
        else:
            from __graft_entry__ import NVCC_FLAGS
            assert torch.cuda.is_available()
            subprocess.check_call([os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")] + NVCC_FLAGS + inc + ["-o", out, PROBE_SRC])
            _PROBES[kind] = Probe(out, kind)
    return _PROBES[kind]


@pytest.fixture(scope="module", params=["cpu", pytest.param(GPU, marks=pytest.mark.gpu)])
def probe(request, tmp_path_factory):
    return _probe(request.param, tmp_path_factory)


@pytest.fixture(scope="module")
def gpu_probe(tmp_path_factory):
    return _probe(GPU, tmp_path_factory)


# ------------------------------------------------------------------ the references: literal chains on Python floats
def binade(e):
    """lo = 2^k and u = 2^(k-52) of e's binade"""
    lo = math.ldexp(0.5, math.frexp(e)[1])
    return lo, math.ldexp(lo, -52)


def literal(e, a, ns, b, npair):
    """ns times e -= a, then npair times (e -= b; e -= a): sub_chain's order"""
    for _ in range(ns):
        e -= a
    for _ in range(npair):
        e -= b
        e -= a
    return e


def tick(e, rr, es, er, nb, ow, na, cap):
    """one node's k+0.5 tick as the reference runs it: nb relays (receive, send), top-up, ow own packets, na relays"""
    e = literal(e, es, 0, er, nb)
    e = min(e + rr * 0.5, cap)
    return literal(e, es, ow, er, na)


def naive_chain(e, a, ns, b, npair):
    """the closed form with the old lower bound r >= lo; None where it would have run the literal loop"""
    lo, u = binade(e)
    qa, qb = a / u, b / u
    ra, rb = round(qa), round(qb)
    if abs(qa - ra) == 0.5 or (npair > 0 and abs(qb - rb) == 0.5):
        return None
    total = ra * (ns + npair) + rb * npair
    r = e - total * u
    return r if total < 2 ** 52 and r >= lo else None


def bits(x):
    return np.asarray(x, np.float64).view(np.uint64)


def step_of(u, r, f):
    """a step of r + f ulps (exact: r < 2^31, f a multiple of 2^-20)"""
    return (float(r) + f) * u


FRACS = {"low": (-0.49, -0.26), "zero": (-0.01, 0.01), "high": (0.26, 0.49)}


def frac(rng, cls):
    lo_f, hi_f = FRACS[cls]
    return math.ldexp(float(rng.integers(int(math.ldexp(lo_f, 20)), int(math.ldexp(hi_f, 20)) + 1)), -20)


def check_chains(probe, cases):
    """cases: (e, a, ns, b, npair).  sub_chain == sub_chain_literal == the Python loop, bit for bit; sub_chain_fast is the same
    value where the closed form is valid (no tie, result strictly above lo) and NaN everywhere else.  Returns the number of
    cases where the old closed form (r >= lo) differs from the literal chain."""
    x = np.array(cases, np.float64)
    want = np.array([literal(*c) for c in cases])
    got = probe(OP_SUB_CHAIN, x)[:, 0]
    got_lit = probe(OP_SUB_CHAIN_LITERAL, x)[:, 0]
    got_fast = probe(OP_SUB_CHAIN_FAST, x)[:, 0]
    for j, c in enumerate(cases):
        assert bits(got[j]) == bits(want[j]), ("sub_chain", c, got[j].hex(), want[j].hex())
        assert bits(got_lit[j]) == bits(want[j]), ("sub_chain_literal", c, got_lit[j].hex(), want[j].hex())
        e, a, ns, b, npair = c
        lo, u = binade(e)
        qa, qb = a / u, b / u
        tie = abs(qa - round(qa)) == 0.5 or (npair > 0 and abs(qb - round(qb)) == 0.5)
        total = round(qa) * (ns + npair) + round(qb) * npair
        valid = ns + npair == 0 or (not tie and total < 2 ** 52 and e - total * u > lo)
        if valid:
            assert bits(got_fast[j]) == bits(want[j]), ("sub_chain_fast", c, got_fast[j].hex(), want[j].hex())
        else:
            assert np.isnan(got_fast[j]), ("sub_chain_fast must decline", c, got_fast[j].hex())
    bad = 0
    for c, w in zip(cases, want):
        nv = naive_chain(*c)
        bad += int(nv is not None and nv != w)
    return bad


def counts():
    return [(ns, npair) for ns in range(9) for npair in range(9) if ns + npair > 0]


# ------------------------------------------------------------------ sub_chain / sub_chain_fast
def test_chains_landing_on_the_binade_floor(probe):
    """chains that end on lo, lo + u and lo + 2u, with the last step's fraction in (-1/2, -1/4), about 0 and in (1/4, 1/2),
    for every n_single / n_pair up to 8"""
    rng = np.random.default_rng(1)
    cases = []
    for k in KS:
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for cls in FRACS:
            for ns, npair in counts():
                ra = int(rng.integers(1, 2_000_000_000))
                rb = int(rng.integers(1, 400_000_000))
                a, b = step_of(u, ra, frac(rng, cls)), step_of(u, rb, frac(rng, "zero"))
                total = ra * (ns + npair) + rb * npair
                for j in range(3):
                    cases.append((lo + (total + j) * u, a, ns, b, npair))
    bad = check_chains(probe, cases)
    assert bad > 0, "no case reached the binade floor with a rounding the old closed form gets wrong"


def test_chains_ties_zero_steps_and_crossings(probe):
    """exact half-ulp ties (literal path), es == 0 (a node without a receiver), steps below half an ulp (ra == 0), and
    chains that cross into the binade below; each with landings on lo"""
    rng = np.random.default_rng(2)
    groups = {"tie": [], "es0": [], "ra0": [], "cross": []}
    for k in KS:
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for ns, npair in counts():
            ra, rb = int(rng.integers(1, 50_000_000)), int(rng.integers(1, 5_000_000))
            total = ra * (ns + npair) + rb * npair
            # ties of a or of b, and near-ties just above 1/4 .. below 1/2, ending on lo .. lo + 2u
            for fa, fb in ((0.5, 0.0), (-0.5, 0.0), (0.0, 0.5), (0.5, -0.5), (0.5 - 2.0 ** -20, 0.0), (0.25 + 2.0 ** -20, 0.0)):
                a, b = step_of(u, ra, fa), step_of(u, rb, fb)
                tot = round(a / u) * (ns + npair) + round(b / u) * npair     # ties to even, as rint
                for j in range(3):
                    groups["tie"].append((lo + (tot + j) * u, a, ns, b, npair))
            # es == 0: only the receive steps move e
            if npair > 0:
                fb = frac(rng, "high")
                for j in range(3):
                    groups["es0"].append((lo + (rb * npair + j) * u, 0.0, ns, step_of(u, rb, fb), npair))
            # a step below half an ulp: nothing moves inside the binade, but at lo the step falls below it
            for fa in (0.3, 0.49, 0.2, 2.0 ** -20):
                for j in range(2):
                    groups["ra0"].append((lo + j * u, fa * u, ns, 0.0, npair))
                    groups["ra0"].append((lo + (rb * npair + j) * u, fa * u, ns, step_of(u, rb, 0.0), npair))
            # crossing: the closed form would end 1 .. 3 ulps below lo (and, for the witness, on lo)
            a = step_of(u, ra, frac(rng, "high"))
            for d in range(0, 4):
                groups["cross"].append((lo + (total - d) * u, a, ns, step_of(u, rb, 0.0), npair))
            groups["cross"].append((lo + (total - ra // 2) * u, a, ns, step_of(u, rb, 0.0), npair))
    for name, cases in groups.items():
        assert check_chains(probe, cases) > 0, name


# ------------------------------------------------------------------ drain_node / replay_cycles
NODES = [  # (nb, ow, na): relays before, own packets, relays after
    (0, 1, 0), (2, 1, 0), (0, 2, 3), (3, 0, 0), (1, 3, 2), (5, 2, 4), (0, 0, 2), (8, 1, 8)]


def node_steps(rng, u, cls):
    es = step_of(u, int(rng.integers(1, 1_000_000_000)), frac(rng, cls))
    er = step_of(u, int(rng.integers(1, 200_000_000)), frac(rng, "zero"))
    return es, er


def K_of(es, er, nb, ow, na, u):
    return round(es / u) * (nb + ow + na) + round(er / u) * (nb + na)


def test_drain_node_and_replay_cycles(probe):
    """drain_node == the literal tick, and replay_cycles == literal cycles, for energies that land on lo with and without a
    top-up, cap inside the binade"""
    rng = np.random.default_rng(3)
    drains, replays, bad = [], [], 0
    for k in KS:
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for nb, ow, na in NODES:
            es, er = node_steps(rng, u, "high")
            K = K_of(es, er, nb, ow, na, u)
            Kb = round(es / u) * nb + round(er / u) * nb
            for rr in (0.0, step_of(u, int(rng.integers(1, 1_000_000)), 0.0) * 2.0):
                for cap in (lo * 1.75, lo + K * u):
                    for e in (lo + K * u, lo + (K + 1) * u, lo + Kb * u, lo + 3 * K * u, lo + (K - 1) * u):
                        drains.append((e, rr, es, er, nb, ow, na, cap))
                        thr = lo - 64.0 * K * u
                        replays.append((e, rr, es, er, nb, ow, na, thr, cap, 5))
                        nv = naive_chain(e, es, ow, er, nb + na) if rr == 0.0 and e <= cap else None
                        bad += int(nv is not None and nv != tick(e, rr, es, er, nb, ow, na, cap))
    got = probe(OP_DRAIN_NODE, drains)[:, 0]
    for g, c in zip(got, drains):
        w = tick(*c)
        assert bits(g) == bits(w), ("drain_node", c, g.hex(), w.hex())
    got = probe(OP_REPLAY_CYCLES, replays)
    for (g, done), c in zip(got[:, :2], replays):
        e, rr, es, er, nb, ow, na, thr, cap, n = c
        want_done = 0
        for _ in range(n):
            e1 = literal(e, es, 0, er, nb)
            if nb > 0 and not (e1 - thr >= SLACK):
                break
            e3 = literal(min(e1 + rr * 0.5, cap), es, ow, er, na)
            if ow + na > 0 and not (e3 - thr >= SLACK):
                break
            e = min(e3 + rr * 0.5, cap)
            want_done += 1
        assert int(done) == want_done and bits(g) == bits(e), ("replay_cycles", c, g.hex(), e.hex(), done, want_done)
    assert bad > 0


# ------------------------------------------------------------------ the table of irregular nodes (spec_terms)
def literal_second(e, node, book, cap):
    rr, es, er, nb, ow, na = node
    if book:
        e = min(e + rr * 0.5, cap)
    return tick(e, rr, es, er, nb, ow, na, cap)


def closed_second(e, t, book, cap):
    """reward_loop's / spec_second's closed form from the entry t = (D1, D2, H, glo, ghi)"""
    D1, D2, H = t[0], t[1], t[2]
    if book:
        e = min(e + H, cap)
    return min((e - D1) + H, cap) - D2


def test_spec_terms_guards(probe):
    """energies at glo - u, glo, glo + u, ghi, ghi + u of an entry, with H == 0 and H > 0 and cap inside the binade: one
    second (drain) and two seconds (drain, then top-up + drain), the closed form inside the guards (rebuilding the entry as
    spec_second does outside them) against the literal seconds.  glo - u is the old lower guard lo + D1 + D2."""
    rng = np.random.default_rng(4)
    bad = {"H0": 0, "H>0": 0}
    n_closed = 0
    for k in KS:
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for nb, ow, na in NODES + [(2, 0, 0), (4, 0, 0)]:
            es, er = node_steps(rng, u, "high")
            D2u = round(es / u) * (ow + na) + round(er / u) * na
            for rr in (0.0, step_of(u, int(rng.integers(1, 1_000_000)), 0.0) * 2.0):
                node = (rr, es, er, nb, ow, na)
                caps = [lo * 1.75]
                if rr > 0.0 and nb == 0:
                    caps.append(lo + D2u * u)          # the top-up clamps to cap and the chain after it ends on lo
                for cap in caps:
                    t = probe(OP_SPEC_TERMS, [(lo * 1.5, es, er, rr, nb, ow, na)])[0]
                    for e in (t[3] - u, t[3], t[3] + u, t[4], t[4] + u):
                        if e > cap:                      # energies never exceed the capacity
                            continue
                        for seconds in ((0,), (0, 1)):
                            want, got, entry = e, e, t
                            for book in seconds:
                                want = literal_second(want, node, book, cap)
                                if entry[3] <= got <= entry[4]:
                                    got = closed_second(got, entry, book, cap)
                                    n_closed += 1
                                else:
                                    got = literal_second(got, node, book, cap)
                                    entry = probe(OP_SPEC_TERMS, [(got, es, er, rr, nb, ow, na)])[0]
                            assert bits(got) == bits(want), (k, node, cap, e.hex(), seconds, got.hex(), want.hex())
                    assert np.isfinite(t[3]) and t[3] == lo + (t[0] + t[1]) + u, (k, node, t)
                    assert t[4] == (lo + lo) - (t[2] + t[2]) - (u + u), (k, node, t)
                    # the old guard: e = lo + D1 + D2 counted as inside
                    e0 = t[3] - u
                    if e0 <= cap:
                        bad["H0" if rr == 0.0 else "H>0"] += int(closed_second(e0, t, 0, cap) != literal_second(e0, node, 0, cap))
    assert n_closed > 0
    assert bad["H0"] > 0 and bad["H>0"] > 0, bad


# ------------------------------------------------------------------ the per-cycle decrement of a whole-cycle batch
def test_batch_decrement(probe):
    """e = lo + j K u (and one or two ulps above) for small j: e - dec m equals m literal cycles and stays above lo; the old
    rule's m = j cycles would land on lo"""
    rng = np.random.default_rng(5)
    rows, meta = [], []
    for k in KS:
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for nb, ow, na in NODES:
            es, er = node_steps(rng, u, "high")
            K = K_of(es, er, nb, ow, na, u)
            for j in range(1, 7):
                for d in range(3):
                    e = lo + (j * K + d) * u
                    for thr in (lo / 2.0, lo + 0.5 * K * u):
                        rows.append((e, es, er, nb, ow, na, thr, 64))
                        meta.append((j, d, K, u, lo))
    got = probe(OP_BATCH_DEC, rows)
    bad, used = 0, 0
    for (dec, m), r, (j, d, K, u, lo) in zip(got[:, :2], rows, meta):
        e, es, er, nb, ow, na, thr, n_max = r
        m = int(m)
        cyc = [e]
        for _ in range(j + 1):
            cyc.append(tick(cyc[-1], 0.0, es, er, nb, ow, na, math.inf))
        if m > 0:
            used += 1
            assert dec == K * u, (r, dec, K)
            assert m <= j, (r, m)
            lit = e
            for _ in range(m):
                lit = tick(lit, 0.0, es, er, nb, ow, na, math.inf)
            assert bits(e - dec * m) == bits(lit) and lit > lo and lit - thr >= SLACK, (r, m, lit.hex())
        else:
            assert np.isnan(dec), (r, dec)
        if d == 0:                                   # the old closed form over j cycles ends on lo
            bad += int(e - K * u * j != cyc[j])
    assert used > 0 and bad > 0, (used, bad)




# ------------------------------------------------------------------ device-only reward helpers against mpmath
def _ulp(x):
    """the spacing of doubles at |x| (normal range)"""
    import mpmath
    return mpmath.ldexp(1, max(int(mpmath.floor(mpmath.log(abs(x), 2))) - 52, -1074))


def _worst(xs, got, exact, rel):
    """largest error of got against exact(x): in ulps of the exact value, or relative (rel=True)"""
    import mpmath
    worst, at = 0.0, None
    for x, g in zip(xs, got):
        ex = exact(mpmath.mpf(float(x)))
        err = abs(mpmath.mpf(float(g)) - ex) / (abs(ex) if rel else _ulp(ex))
        if err > worst:
            worst, at = float(err), float(x)
    return worst, at


def _mantissa_edges(e_lo, e_hi):
    return [math.ldexp(m, ex) for ex in range(e_lo, e_hi) for m in (1.0, 1.0 + 2.0 ** -52, 2.0 - 2.0 ** -52)]


@pytest.mark.gpu
def test_device_reward_helpers_against_mpmath(gpu_probe):
    """wrsn_rcp / wrsn_rsqrt within 2 ulp (d > 0 with d and the result normal), wrsn_exp_tab within 1e-13 relative for
    |z| < 700: mantissas 1, 1 + ulp, 2 - ulp at every exponent, the ends of the normal range, random inputs; z on and next to
    every table boundary j ln2/64 and every switch point (j + 1/2) ln2/64 the caller reaches (|z| <= sqrt(1151)), a sparse
    set of them up to 700, and random z"""
    import mpmath
    mpmath.mp.dps = 50
    rng = np.random.default_rng(6)
    dmin, dmax = np.finfo(np.float64).tiny, np.finfo(np.float64).max
    ends = [dmin, np.nextafter(dmin, 1.0), dmin * 2.0, np.nextafter(dmin * 2.0, 0.0), dmax, np.nextafter(dmax, 0.0),
            2.0 ** 1022, np.nextafter(2.0 ** 1022, 0.0)]
    rand = list(np.exp2(rng.uniform(-1022.0, 1023.0, 20000)))
    report = {}
    # rcp: the result must be normal too, d <= 2^1022
    xs = [x for x in _mantissa_edges(-1022, 1023) + ends + rand if x <= 2.0 ** 1022]
    report["rcp"] = _worst(xs, gpu_probe(OP_RCP, xs)[:, 0], lambda x: 1 / x, False)
    big = [x for x in _mantissa_edges(1022, 1024) + ends if x > 2.0 ** 1022]
    report["rcp beyond 2^1022 (not bounded)"] = _worst(big, gpu_probe(OP_RCP, big)[:, 0], lambda x: 1 / x, False)
    xs = _mantissa_edges(-1022, 1024) + ends + rand
    report["rsqrt"] = _worst(xs, gpu_probe(OP_RSQRT, xs)[:, 0], lambda x: 1 / mpmath.sqrt(x), False)
    step = math.log(2.0) / 64.0
    zs = []
    for j in list(range(-3200, 3201)) + list(range(-64640, 64641, 97)):
        for z0 in (j * step, (j + 0.5) * step):
            if abs(z0) < 700.0:
                zs += [np.nextafter(z0, -math.inf), z0, np.nextafter(z0, math.inf)]
    zs += [math.sqrt(n - 1.0) * s for n in range(1, 1153) for s in (1.0, -1.0)]
    zs += [np.nextafter(700.0, 0.0), np.nextafter(-700.0, 0.0)] + list(rng.uniform(-700.0, 700.0, 20000))
    report["exp_tab"] = _worst(zs, gpu_probe(OP_EXP_TAB, zs)[:, 0], mpmath.exp, True)
    print("worst errors (value, at input):", report)
    assert report["rcp"][0] <= 2.0 and report["rsqrt"][0] <= 2.0 and report["exp_tab"][0] <= 1e-13, report


# ------------------------------------------------------------------ end to end: the engine and the C oracle at binade edges
NET = "net_hanoi1000n50"
T0 = 300.0


@pytest.fixture(scope="module")
def emu_built():
    subprocess.check_call(["make", "-C", EMU_DIR, "libwrsn_emu.so"], stdout=subprocess.DEVNULL)


@pytest.fixture
def dev(request, emu_built):
    """The host emulation for "cpu", the CUDA library (no fallback) for the GPU."""
    if request.param == "cpu":
        helpers.use_host_build()
        yield "cpu"
        helpers.use_cuda_build_lazy()
    else:
        L = helpers.use_cuda_build()
        assert not helpers.is_host_build(L) and torch.cuda.is_available()
        yield request.param


DEVS = ["cpu", pytest.param(GPU, marks=pytest.mark.gpu)]


def edge_nodes(env, o, row=0, skip=()):
    """alive, uncharged nodes with traffic, each with the lowest binade 2^k in (threshold, capacity) in which the last
    subtraction of its tick has a fraction above 1/4 (no tie): {i: (lo, u, K)}, K = ulps per tick"""
    p = env.statics[0]["par"]
    thr, cap, er = p["THR"], p["CAP"], p["ERECV"]
    es, rr = pc._np(env.view("esend"))[row], pc._np(env.view("rr"))[row]
    nb, na = pc._np(env.view("nbef"))[row].astype(int), pc._np(env.view("naft"))[row].astype(int)
    par, st = pc._np(env.view("parent"))[row].astype(int), pc._np(env.view("status"))[row]
    own = np.diff(o.static_graph()["tgt_ptr"])
    out = {}
    for i in range(env.N):
        ow = int(own[i]) if par[i] != -1 else 0
        if st[i] != 1 or rr[i] != 0.0 or nb[i] + ow + na[i] == 0 or i in skip:
            continue
        for k in range(math.floor(math.log2(thr)) + 1, math.floor(math.log2(cap)) + 1):
            lo, u = 2.0 ** k, 2.0 ** (k - 52)
            qa, qb = es[i] / u, er / u
            ra, rb = round(qa), round(qb)
            last = qa - ra if es[i] > 0.0 and (ow + na[i] > 0 or nb[i] > 0) else qb - rb
            if 0.25 < last < 0.5 and abs(qa - ra) != 0.5 and abs(qb - rb) != 0.5:
                out[i] = (lo, u, ra * (nb[i] + ow + na[i]) + rb * (nb[i] + na[i]))
                break
    return out


def same_nodes(env, o, tag, row=0):
    nd = o.nodes()
    assert np.array_equal(pc._np(env.view("status"))[row], nd["status"]), tag
    e = pc._np(env.view("energy"))[row]
    diff = np.nonzero(bits(e) != bits(nd["energy"]))[0]
    assert diff.size == 0, (tag, [(int(i), e[i].hex(), nd["energy"][i].hex()) for i in diff[:5]])
    assert np.array_equal(bits(pc._np(env.view("cs"))[row]), bits(nd["cs"])), tag


def pure_network(device):
    sc = pc.sc_from_golden(helpers.golden(NET))
    env = pc.BatchedWRSN(sc, num_agent=0, num_envs=1, device=device)
    env.init_network(with_reward_process=False)
    o = pc.OracleWRSN(pc.scenario_from_dict(sc.to_dict()), num_agent=0)
    o.start_network_only()
    env.run_until(T0 + 0.25)
    o.run_until(T0 + 0.25)
    same_nodes(env, o, "start")
    return env, o


def put_energy(env, o, i, e, row=0):
    env.view("energy")[row, i] = e
    o.set_node_energy(i, e)


@pytest.mark.parametrize("dev", DEVS, indirect=True)
def test_drain_tick_lands_on_binade_floor(dev):
    """energies 2^k + K u: the drain tick ends exactly on 2^k, where the reference rounds to 2^k - u/2"""
    env, o = pure_network(dev)
    nodes = edge_nodes(env, o)
    assert len(nodes) >= 20, len(nodes)
    for i, (lo, u, K) in nodes.items():
        put_energy(env, o, i, lo + K * u)
    env.kernel("drain")
    o.run_until(T0 + 0.75)
    same_nodes(env, o, "drain")
    e = o.nodes()["energy"]
    assert all(e[i] == lo - u / 2 for i, (lo, u, K) in nodes.items())


@pytest.mark.parametrize("dev", DEVS, indirect=True)
def test_batches_and_event_ticks_land_on_binade_floor(dev):
    """energies 2^k + j K u, j = 1 .. 30: 40 s of whole-cycle batches, cycle replays and event ticks, each node landing on
    2^k at its j-th tick"""
    env, o = pure_network(dev)
    nodes = edge_nodes(env, o)
    assert len(nodes) >= 20, len(nodes)
    land = {}
    for n, (i, (lo, u, K)) in enumerate(sorted(nodes.items())):
        j = 1 + n % 30
        put_energy(env, o, i, lo + j * K * u)
        land[i] = j
    env.run_until(T0 + 40.0)
    reached = set()
    for s in range(40):
        o.run_until(T0 + s + 0.75)
        e = o.nodes()["energy"]
        reached |= {i for i, j in land.items() if j == s + 1 and e[i] == nodes[i][0] - nodes[i][1] / 2}
    o.run_until(T0 + 40.0)
    same_nodes(env, o, "run_until")
    assert len(reached) >= 0.9 * len(land), (len(reached), len(land))


@pytest.mark.parametrize("dev", DEVS, indirect=True)
def test_active_batch_lands_on_binade_floor(dev):
    """one charger parked for a long charge (update_reward active: the batches keep a table of irregular nodes), the other
    re-sent to the same spot; at a request, far uncharged nodes get 2^k + j K u (j = 1 .. 4: the old lower guard of the table,
    2^k + D1 + D2, after j - 1 ticks) in both simulators; then on to the next requests"""
    sc = pc.sc_from_golden(helpers.golden(NET))
    env = pc.BatchedWRSN(sc, num_agent=2, num_envs=1, device=dev)
    o = pc.OracleWRSN(pc.scenario_from_dict(sc.to_dict()), num_agent=2)
    req, r = env.reset(), o.reset(want_state=False)
    f = o.consts()["frame"]
    xy = o.sc["nodes"]
    spot = xy[np.argmin(np.hypot(xy[:, 0] - (f[0] + f[1]) / 2, xy[:, 1] - (f[2] + f[3]) / 2))]
    ax, ay = (spot[0] - f[0]) / (f[1] - f[0]), (spot[1] - f[2]) / (f[3] - f[2])
    park, short = np.array([ax, ay, 1.0]), np.array([ax, ay, 0.02])
    crafted, charged = {}, 0
    for k in range(8):
        aid = int(pc._np(req.agent_id)[0])
        assert aid == r["raw_agent_id"] and aid >= 0, k
        assert int(pc._np(req.terminal)[0]) == int(r["terminal"]) and float(pc._np(req.now)[0]) == r["now"], k
        if k > 0 and k != 3:                         # the reward of the step across the write differs by design: the
            # engine's reward takes the energies before the write, the oracle's after it
            np.testing.assert_allclose(float(pc._np(req.reward)[0]), r["reward"], rtol=1e-9, atol=1e-18)
        same_nodes(env, o, ("request", k))
        charged += int((o.nodes()["rr"] > 0.0).any())
        if k == 2:
            nodes = edge_nodes(env, o)
            for n, (i, (lo, u, K)) in enumerate(sorted(nodes.items())[:12]):
                put_energy(env, o, i, lo + (1 + n % 4) * K * u)
                crafted[i] = (lo, u)
        act = park if k == 0 else short
        req = env.step(np.array([aid], np.int32), act[None, :])
        r = o.step(aid, act, want_state=False)
    assert len(crafted) >= 8 and charged >= 6, (len(crafted), charged)
    e = o.nodes()["energy"]
    assert all(e[i] < lo for i, (lo, u) in crafted.items())     # every crafted node has crossed its 2^k
