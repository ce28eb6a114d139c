"""The lazy charger spans' closed forms at energy-binade, threshold and time-binade edges, against literal per-second replays.

A charger that charges where no alive node is in range, or moves far from its destination, repeats one private event per
second; the engine replays such a run in registers (``slot_ff``).  Two of its shortcuts have edges of their own:

- ``charge_run`` applies m one-second charge spans at once: the energy drops by m rint(rate / u) ulps of its binade (ties
  refused), m is cut one span before the binade floor or the charger's threshold (``floor(room / (rq u)) - 1``), before the
  next power of two of the event time (where adding 1.0 may round) and before the replay's time limit, and the countdowns drop
  by m (CPA2 clamped at 0);
- ``move_span_is_one`` takes a move span as 1 s without the square root when ``d2 > v^2 1.000001`` and
  ``en1 - thr >= pm v``; that is right only if the literal ``sqrt(d2) / v`` is then > 1, so that the skipped arrival check
  could not have fired.

``tests/emu/energy_probe.cu`` exposes both, for the host build and (``-m gpu``) the device; the reference is the reference's
per-second loop on Python floats (IEEE doubles), compared bit for bit with jumps on and off.  Every group also runs a Python
restatement of ``charge_run`` with a named change (a mutant) and fails unless at least one of its cases makes the mutant differ
from the literal loop, so the cases reach the edge that guard protects:

- M1: ``floor(room / (rq u))`` without the ``- 1``;  M2: ``room = en - lo`` (threshold ignored);  M3: no tie refusal;
- M4: no time-binade cap;  M5: no ``floor(limit - tf)`` cap;  M6: ``far = v * v``;
- C1: ``m = tmp`` for an integral remaining time (the last span included);  C2: ``cpa2 - m`` without the clamp at 0.

Changes that stay correct and pass are not mutants: ``en1 - thr > pmv``, or a margin of ``- 2.0`` instead of ``- 1.0`` (the
jump is only shorter).

End to end, crafted charger energies just above a power of two, a threshold above the binade floor and warm-ups just below
2^11, 2^12 and 2^13 s drive the lazy charges through the same edges inside the engine: against the C oracle bit for bit, with
the jumps on and off byte for byte, and cut by the ends of launches under step budgets of 1 .. 7.  Each case counts its regimes
from the record at every request and fails below a floor."""
import dataclasses
import math
import os
import re

import numpy as np
import pytest
import torch

from multi_agent_rl_wrsn_b200 import synthetic
from multi_agent_rl_wrsn_b200.scenario import DEFAULT_MC
from tests import helpers
from tests import parity_cases as pc
from tests.test_energy_chains import DEVS, GPU, OP_CHARGE_RUN, OP_MOVE_SPAN, _probe, bits
from tests.test_energy_chains import dev, emu_built  # noqa: F401  (fixtures)

INF = math.inf
TWO52 = 2.0 ** 52


@pytest.fixture(scope="module", params=["cpu", pytest.param(GPU, marks=pytest.mark.gpu)])
def probe(request, tmp_path_factory):
    return _probe(request.param, tmp_path_factory)


# ------------------------------------------------------------------ the references
def on_grid(t):
    f = float(math.floor(t))
    return t == f or t == f + 0.5 or t == f + 0.1


def _floor(x):
    return x if math.isinf(x) else float(math.floor(x))


def literal_run(en, rate, thr, tmp, cpa2, span, tf, limit):
    """the reference's charge spans one second at a time (charge_step :45-46, charge :63-69): spans whose event time is below
    ``limit``, up to a span on the node grid, the end of the charge or exhaustion -> (en, cpa2, tmp, span, tf, n, t_end)"""
    n, t_end = 0, INF
    while tf < limit:
        if on_grid(tf):
            t_end = tf
            break
        en1 = en - rate * span
        cpa21 = max(0.0, cpa2 - span)
        tmp1 = tmp - span
        if tmp1 == 0.0 or en1 <= thr:
            t_end = tf
            break
        en, cpa2, tmp, span = en1, cpa21, tmp1, min(tmp1, 1.0)
        tf = tf + span
        n += 1
    return en, cpa2, tmp, span, tf, n, t_end


def model_run(en, rate, thr, tmp, cpa2, span, tf, limit, mutant=None, jumped=None):
    """charge_run with jumps, restated line by line; ``mutant`` names one change of the list above.  ``jumped``: a list that
    receives the length of every jump taken."""
    n, t_end = 0, INF
    while tf < limit:
        if on_grid(tf):
            t_end = tf
            break
        if span == 1.0 and 2.0 < tmp < 2.0 ** 30 and cpa2 < TWO52:
            fl = float(math.floor(tmp))
            m = tmp - 1.0 if fl == tmp and mutant != "C1" else fl
            if mutant != "M5":
                m = min(m, _floor(limit - tf))
            ext = math.frexp(tf)[1] + 1022                  # the biased exponent of tf
            if tf > 0.0 and 60 < ext < 1100:
                if mutant != "M4":
                    m = min(m, _floor(math.ldexp(1.0, ext - 1022) - tf))
            else:
                m = 0.0
            en_m = en
            if rate != 0.0:
                ex = math.frexp(en)[1] + 1022
                if en > 0.0 and 60 < ex < 1900:
                    lo, u = math.ldexp(1.0, ex - 1023), math.ldexp(1.0, ex - 1075)
                    q = rate / u
                    rq = float(round(q))                      # ties to even, as rint
                    room = en - (lo if mutant == "M2" else max(lo, thr))
                    if (abs(q - rq) == 0.5 and mutant != "M3") or not rq > 0.0 or not room > 0.0:
                        m = 0.0
                    else:
                        m = min(m, _floor(room / (rq * u)) - (0.0 if mutant == "M1" else 1.0))
                        if m >= 2.0 and rq * m < TWO52:
                            en_m = en - (rq * m) * u
                        else:
                            m = 0.0
                else:
                    m = 0.0
            if m >= 2.0:
                en = en_m
                cpa2 = cpa2 - m if cpa2 >= m or mutant == "C2" else 0.0
                tmp = tmp - m
                span = min(tmp, 1.0)
                tf = (tf + (m - 1.0)) + span
                n += int(m)
                if jumped is not None:
                    jumped.append(int(m))
                continue
        en1 = en - rate * span
        cpa21 = max(0.0, cpa2 - span)
        tmp1 = tmp - span
        if tmp1 == 0.0 or en1 <= thr:
            t_end = tf
            break
        en, cpa2, tmp, span = en1, cpa21, tmp1, min(tmp1, 1.0)
        tf = tf + span
        n += 1
    return en, cpa2, tmp, span, tf, n, t_end


def _same(a, b):
    return all(bits(x) == bits(y) for x, y in zip(a, b))


def check_runs(probe, cases, mutants):
    """cases: (en, rate, thr, tmp, cpa2, span, tf, limit).  The probe with jumps on and off, and the restatement, equal the
    literal loop bit for bit.  Returns ({mutant: cases where it differs from the literal loop}, jumps taken)."""
    rows = np.array([c + (j,) for c in cases for j in (1.0, 0.0)], np.float64)
    got = probe(OP_CHARGE_RUN, rows)
    caught = {mu: 0 for mu in mutants}
    jumps = 0
    for i, c in enumerate(cases):
        want = literal_run(*c)
        for j in range(2):
            y = got[2 * i + j]
            g = (y[0], y[1], y[2], y[3], y[4], y[6], y[7])
            assert _same(g, want), ("charge_run", "jumps" if j == 0 else "literal", [float(v).hex() for v in c],
                                    [float(v).hex() for v in g], [float(v).hex() for v in want])
        jumped = []
        assert _same(model_run(*c, jumped=jumped), want), ("restatement", c)
        jumps += int(len(jumped) > 0)
        for mu in mutants:
            caught[mu] += int(not _same(model_run(*c, mutant=mu), want))
    return caught, jumps


def assert_caught(caught, jumps, group):
    assert jumps > 0, (group, "no case took a jump")
    missing = [mu for mu, k in caught.items() if k == 0]
    assert not missing, (group, "no case tells these mutants from the literal loop", missing, caught)
    print(group, "jumps", jumps, "mutant witnesses", caught)


def binade(e):
    lo = math.ldexp(0.5, math.frexp(e)[1])
    return lo, math.ldexp(lo, -52)


def rate_of(u, r, f):
    """a rate of r + f ulps (exact: r < 2^31, f a multiple of 2^-20)"""
    return (float(r) + f) * u


FRACS = {"low": (-0.49, -0.26), "zero": (-0.01, 0.01), "high": (0.26, 0.49)}


def frac(rng, cls):
    lo_f, hi_f = FRACS[cls]
    return math.ldexp(float(rng.integers(int(math.ldexp(lo_f, 20)), int(math.ldexp(hi_f, 20)) + 1)), -20)


TF0 = 300.25                                         # off the node grid, far from a power of two
TMP0 = 30.5


# ------------------------------------------------------------------ the groups
def test_energy_binade(probe):
    """en = 2^k + j rq u + d for j around the cap (1 .. 9) and d = 0, 1, 2, rq / 2, rq - 1 ulps, k = 3 .. 17; rate fractions
    in (-1/2, -1/4), about 0, in (1/4, 1/2) and exactly +-1/2 (ties); rate 0 and rates below u / 2"""
    rng = np.random.default_rng(11)
    cases = []
    for k in range(3, 18):
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for cls in ("low", "zero", "high", 0.5, -0.5):
            r = int(rng.integers(2, 2 ** 31 // 16))
            f = cls if isinstance(cls, float) else frac(rng, cls)
            rate = rate_of(u, r, f)
            rq = round(rate / u)
            for j in range(1, 10):
                for d in (0, 1, 2, rq // 2, rq - 1):
                    cases.append((lo + float(j * rq + d) * u, rate, 0.0, TMP0, 20.0, 1.0, TF0, INF))
        for rate in (0.0, 0.3 * u, 0.49 * u, 0.26 * u, 0.5 * u, math.ldexp(u, -20)):
            for en in (lo, lo + u, lo + 2 * u, lo * 1.5):
                cases.append((en, rate, 0.0, TMP0, 20.0, 1.0, TF0, INF))
    caught, jumps = check_runs(probe, cases, ("M1", "M3"))
    assert_caught(caught, jumps, "energy binade")


def test_threshold(probe):
    """thr = 0; lo < thr < en; thr exactly at en - m rq u (the end of a jump); thr = lo; exhaustion one span inside and one
    span outside the jump window, and on either side of the threshold by an ulp"""
    rng = np.random.default_rng(12)
    cases = []
    for k in range(3, 18):
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        for cls in ("low", "zero", "high"):
            rate = rate_of(u, int(rng.integers(2, 2 ** 31 // 16)), frac(rng, cls))
            rq = round(rate / u)
            thr_in = lo + float(int(rng.integers(1, 2 ** 40))) * u          # lo < thr, far below 2 lo
            for j in range(1, 8):
                for thr in (0.0, lo, thr_in):
                    base = max(lo, thr)
                    for d in (0, 1, rq - 1):
                        cases.append((base + float(j * rq + d) * u, rate, thr, TMP0, 20.0, 1.0, TF0, INF))
                # the threshold exactly where a jump of m spans ends, and an ulp either side of it
                en = thr_in + float(j * rq) * u
                for m in (j - 1, j, j + 1):
                    t = en - float(m * rq) * u
                    for tt in (t, np.nextafter(t, 0.0), np.nextafter(t, INF)):
                        if 0.0 < tt < en:
                            cases.append((en, rate, float(tt), TMP0, 20.0, 1.0, TF0, INF))
            # exhaustion just inside / just outside the jump window: the charge ends (tmp) one span before, at, or after
            # the span that would cross the threshold
            for j in (3, 5, 8):
                en = thr_in + float(j * rq + 1) * u
                for tmp in (j - 1.0, float(j), j + 1.0, j + 0.5, j - 0.5):
                    cases.append((en, rate, thr_in, tmp, 20.0, 1.0, TF0, INF))
                for lim in (TF0 + j - 1.0, TF0 + j, TF0 + j + 1.0):
                    cases.append((en, rate, thr_in, TMP0, 20.0, 1.0, TF0, lim))
    caught, jumps = check_runs(probe, cases, ("M1", "M2"))
    assert_caught(caught, jumps, "threshold")


def test_time_binade_and_limit(probe):
    """tf crossing 2^11 .. 2^15 with fractions .0, .5, f + 0.1, .25 and one to three ulps off them; limit at +inf, at an
    integer distance from tf, within an ulp of it on either side, and below tf"""
    rng = np.random.default_rng(13)
    cases = []
    for k in range(11, 16):
        lo, u = 2.0 ** 16, 2.0 ** (16 - 52)
        rate = rate_of(u, int(rng.integers(2, 2 ** 20)), frac(rng, "zero"))
        en = lo * 1.5                                            # far from the energy's binade floor
        for d in range(1, 7):
            base = float(2 ** k - d)
            grids = [base, base + 0.5, base + 0.1, base + 0.25]
            for t0 in grids:
                tfs = [t0]
                for s in (1, 2, 3):
                    tfs += [t0 + s * math.ulp(t0), t0 - s * math.ulp(t0)]
                for tf in tfs:
                    for lim in (INF, tf + 4.0, tf + 9.0, np.nextafter(tf + 4.0, 0.0), np.nextafter(tf + 4.0, INF), tf - 1.0,
                                float(2 ** k) + 2.5):
                        cases.append((en, rate, 0.0, TMP0, 20.0, 1.0, tf, float(lim)))
                    cases.append((en, 0.0, 0.0, TMP0, 20.0, 1.0, tf, INF))
    caught, jumps = check_runs(probe, cases, ("M4", "M5"))
    assert_caught(caught, jumps, "time")


def test_countdowns(probe):
    """integral and fractional remaining times, tmp in (2, 3], tmp near 2^30; CPA2 below the jump's m, equal to it, above it
    and 0; a first span shorter than 1 s"""
    rng = np.random.default_rng(14)
    cases = []
    for k in (5, 9, 13, 17):
        lo, u = 2.0 ** k, 2.0 ** (k - 52)
        rate = rate_of(u, int(rng.integers(2, 2 ** 20)), frac(rng, "high"))
        en = lo * 1.5
        tmps = [3.0, 7.0, 50.0, 2.0, 2.5, 3.0, np.nextafter(2.0, INF), np.nextafter(3.0, 0.0), 7.3, 50.5, 12.1,
                2.0 ** 30 - 1.0, 2.0 ** 30 - 0.5, 2.0 ** 30, 2.0 ** 30 + 0.5, np.nextafter(2.0 ** 30, 0.0)]
        for tmp in tmps:
            tmp = float(tmp)
            lim = TF0 + 80.0 if tmp > 100 else INF
            m = float(math.floor(tmp)) - (1.0 if math.floor(tmp) == tmp else 0.0)    # the jump the energy does not cut
            m = min(m, 80.0) if tmp > 100 else m
            for cpa2 in (0.0, m - 1.0, m, m + 1.0, m - 0.5, m + 0.5, 1.5, 2.0 ** 52 - 1.0, 2.0 ** 52):
                if cpa2 >= 0.0:
                    cases.append((en, rate, 0.0, tmp, cpa2, 1.0, TF0, lim))
            cases.append((en, rate, 0.0, tmp, 5.0, 0.5, TF0, lim))
            cases.append((en, rate, 0.0, tmp, 5.0, 0.25, TF0 + 0.25, lim))
    caught, jumps = check_runs(probe, cases, ("C1", "C2"))
    assert_caught(caught, jumps, "countdowns")


def move_span_ref(d2, en1, thr, v, pmv, far_of=lambda v: v * v * 1.000001):
    return d2 > far_of(v) and en1 - thr >= pmv


def test_move_shortcut(probe):
    """d2 at and one ulp around v^2, v^2 1.000001 and v^2 (1 + 1e-7); en1 - thr at, and one to three ulps below and above,
    pm v.  Wherever the shortcut fires, the literal span min(mt, 1, (en1 - thr) / pmv) is 1.0 and mt - 1.0 > 0 (the arrival
    check it skips stays false); far from both edges it fires."""
    rng = np.random.default_rng(15)
    rows = []
    for v in [5.0, 1.0, 0.1, 7.3, 100.0, 3.0] + list(rng.uniform(0.05, 50.0, 40)):
        for pm in (1.0, 0.5, 3.7):
            pmv = pm * v
            thr = float(rng.choice([0.0, 10.0, 540.25]))
            vv, far = v * v, v * v * 1.000001
            d2s = []
            for c in (vv, far, 4.0 * vv, vv * (1.0 + 1e-7)):
                d2s += [c, np.nextafter(c, 0.0), np.nextafter(c, INF), np.nextafter(np.nextafter(c, INF), INF)]
            en1s = []                                # en1 - thr rounds: walk en1 by ulps around thr + pmv
            for e in (thr + pmv, thr + pmv * 10.0):
                for s in range(-3, 4):
                    x = e
                    for _ in range(abs(s)):
                        x = np.nextafter(x, INF if s > 0 else 0.0)
                    en1s.append(float(x))
            for d2 in d2s:
                for en1 in en1s:
                    rows.append((float(d2), en1, thr, v, pmv))
    got = probe(OP_MOVE_SPAN, rows)[:, 0]
    fired = clear = edge = caught = 0
    for g, (d2, en1, thr, v, pmv) in zip(got, rows):
        mt = math.sqrt(d2) / v
        literal_one = min(min(mt, 1.0), (en1 - thr) / pmv) == 1.0 and mt - 1.0 > 0.0
        if g:
            fired += 1
            assert literal_one, ("the shortcut fires where the literal span is not a full second", d2.hex(), en1.hex(), thr, v, pmv)
            edge += int(en1 - thr == pmv)
        if d2 >= 4.0 * v * v and en1 - thr >= 10.0 * pmv:
            clear += 1
            assert g, ("the shortcut must fire far from the destination and from exhaustion", d2.hex(), en1.hex(), v)
        caught += int(move_span_ref(d2, en1, thr, v, pmv, far_of=lambda v: v * v) and not literal_one)
    assert fired > 0 and clear > 0, (fired, clear)
    assert caught > 0, "no case tells M6 (far = v * v) from the literal arithmetic"
    print("move shortcut: fired", fired, "of", len(rows), "(at en1 - thr == pmv:", edge, ") M6 witnesses", caught)


# ------------------------------------------------------------------ end to end: crafted charger energies, engine vs C oracle
# a small charger type whose threshold lies above the floor of the binade [256, 512) it charges in; cheap moves, so that it
# can charge the nodes around the base station without running dry on the way back
MC_THR = dict(DEFAULT_MC, capacity=700.0, threshold=300.0, pm=0.25)
E_FLOOR = 512.0                                      # the crafted energies sit above this power of two


def _pc_cs_fire():
    """the program counter of a pending charge span (the slot enum of wrsn_engine.cuh)"""
    with open(os.path.join(helpers.REPO, "multi_agent_rl_wrsn_b200", "csrc", "wrsn_engine.cuh")) as f:
        src = f.read()
    names = re.search(r"PC_OP_INIT = 1,([^}]*)}", src).group(1).replace(",", " ").split()
    return 2 + names.index("PC_CS_FIRE")


def _exp(x):
    return np.frexp(x)[1]


class LazyWitness:
    """Counts, from the record at every request, the regimes of the lazy charge runs (rows x requests):
    nlazy = NLAZY grew; binade = a charge slot lazy at this request, with owed insertion counters, whose charger's energy is in
    another binade than at the previous request (after the edits); time = the same with ``now`` across a power of two; tie = a
    lazy charge whose rate is an exact half-ulp tie of its charger's energy; thr_lo = a lazy charge whose charger's energy lies in
    a binade whose floor is below the threshold."""

    def __init__(self, thr):
        self.thr, self.cs = thr, _pc_cs_fire()
        self.n = dict(nlazy=0, binade=0, time=0, tie=0, thr_lo=0)
        self.prev = None

    def _lazy_cs(self, env):
        E = env.E
        pi = env.view("proc").view(torch.int32)
        lazy = pi[:, :, E["WRSN_PRI_LAZY"]].cpu().numpy() != 0
        pcs = pi[:, :, E["WRSN_PRI_PC"]].cpu().numpy()
        agent = pi[:, :, E["WRSN_PRI_AGENT"]].cpu().numpy()
        owed = pc._np(env.view("proc")[:, :, E["WRSN_PR_OWED"]])
        return lazy & (pcs == self.cs) & (owed > 0.0), agent

    def probe(self, env, live):
        run, agent = self._lazy_cs(env)
        en, rate = pc._np(env.mc("ENERGY")), pc._np(env.mc("RATE"))
        now, nlazy = pc._np(env.now), pc._np(env.hdr("NLAZY"))
        for b in np.nonzero(live)[0]:
            if self.prev is not None:
                self.n["nlazy"] += int(nlazy[b] > self.prev["nlazy"][b])
            for s in np.nonzero(run[b])[0]:
                a = int(agent[b, s])
                e, r = float(en[b, a]), float(rate[b, a])
                lo, u = binade(e)
                q = r / u
                self.n["tie"] += int(r > 0.0 and abs(q - round(q)) == 0.5)
                self.n["thr_lo"] += int(lo < self.thr)
                if self.prev is not None:
                    self.n["binade"] += int(_exp(e) != _exp(self.prev["en"][b, a]))
                    self.n["time"] += int(_exp(now[b]) != _exp(self.prev["now"][b]))
        self.prev = dict(nlazy=nlazy, en=en, now=now)

    def edited(self, b, a, e):
        self.prev["en"][b, a] = e


def _normalised(env, b, x, y):
    par = env.statics[int(pc._np(env.scen_id)[b])]["par"]
    return (x - par["F0"]) / (par["F1"] - par["F0"]), (y - par["F2"]) / (par["F3"] - par["F2"])


def crafted_charges(offsets, seed):
    """``plan(env, live, aid, act)``, before every step: the deciding charger of row b goes to one of the 8 alive nodes nearest
    to the base station (the same choice in every row) for a charge of 16 .. 62 s, with its
    energy set to E_FLOOR + (the energy its move costs) + offsets[b].  Writes the actions and the energies into ``act`` and
    ``env``, and returns the edits [(row, charger, energy)].  Only the decider is edited: a lazy slot's end (TINT) was found
    from its charger's energy."""
    rng = np.random.default_rng(seed)

    def plan(env, live, aid, act):
        spe = env.scenarios[0].node_phy_spe
        ct_max = (spe["capacity"] - spe["threshold"]) / (MC_THR["alpha"] / MC_THR["beta"] ** 2)    # WRSN.charging_time_max
        pick, frac_ct = int(rng.integers(0, 8)), float(rng.uniform(16.0, 62.0)) / ct_max
        st, mx, my = pc._np(env.view("status")), pc._np(env.mc("X")), pc._np(env.mc("Y"))
        sid = pc._np(env.scen_id)
        edits = []
        for b in np.nonzero(live & (aid >= 0))[0]:
            a, sc = int(aid[b]), env.scenarios[sid[b]]
            xy, bs = np.asarray(sc.nodes, np.float64), np.asarray(sc.base_station, np.float64)
            d = np.hypot(xy[:, 0] - bs[0], xy[:, 1] - bs[1])
            d[st[b][:len(d)] != 1] = np.inf
            dest = xy[np.argsort(d, kind="stable")[pick]]
            act[b, 0], act[b, 1] = _normalised(env, b, dest[0], dest[1])
            act[b, 2] = frac_ct
            move = float(np.hypot(dest[0] - mx[b, a], dest[1] - my[b, a])) * MC_THR["pm"]
            e = E_FLOOR + move + float(offsets[b])
            env.mc("ENERGY")[b, a] = e
            edits.append((b, a, e))
        return edits
    return plan


def field():
    """the 50-node Hanoi field with nodes of 8 times the capacity, so that the network outlives a warm-up of 2^13 s"""
    sc = pc.sc_from_golden(helpers.golden("ep_deadmc_n50"))
    return dataclasses.replace(sc, node_phy_spe=dict(sc.node_phy_spe, capacity=8.0 * sc.node_phy_spe["capacity"]))


def _offsets(rows):
    return np.linspace(-20.0, 160.0, rows) + np.linspace(0.0, 0.37, rows)       # one row per offset


def lazy_charges_vs_oracle(dev, warm_up, rows, steps, seed):
    sc = field()
    w = LazyWitness(MC_THR["threshold"])
    plan = crafted_charges(_offsets(rows), seed)

    def before_step(env, oracles, k, live, aid, act):
        for b, a, e in plan(env, live, aid, act):
            oracles[b].set_mc_energy(a, e)
            w.edited(b, a, e)
    n_dec, cnt = pc.check_vs_oracle(sc, dev, num_envs=rows, steps=steps, seed=seed, num_agent=3, mc=MC_THR, scale2=1.0,
                                    probe=w.probe, warm_up_time=warm_up, before_step=before_step)
    return n_dec, cnt, w.n


WARM_UPS = [2.0 ** 11 - 37.25, 2.0 ** 12 - 61.75, 2.0 ** 13 - 23.5]


@pytest.mark.parametrize("dev", DEVS, indirect=True)
def test_lazy_charges_at_energy_and_time_binades_vs_oracle(dev):
    """At every request the deciding charger (a 700 J type with a 300 J threshold) gets an energy just above 512 J plus its
    move, one row per offset, and goes to charge a node near it for up to the longest charge; warm-ups just below 2^11, 2^12
    and 2^13 s, so that its lazy charges cross the energy's and the clock's powers of two.  Every row at every request against
    the C oracle, bit for bit; the regimes are counted from the record and must all be reached."""
    total = dict(nlazy=0, binade=0, time=0, tie=0, thr_lo=0)
    n_all = 0
    for i, wu in enumerate(WARM_UPS):
        n_dec, cnt, n = lazy_charges_vs_oracle(dev, wu, rows=8, steps=30, seed=40 + i)
        n_all += n_dec
        for key in total:
            total[key] += n[key]
    print("lazy charges vs oracle: decisions", n_all, "witnesses", total)
    assert n_all >= 600, n_all
    assert (total["nlazy"] >= 400 and total["binade"] >= 150 and total["time"] >= 20 and total["tie"] >= 10
            and total["thr_lo"] >= 200), total


@pytest.mark.parametrize("dev", DEVS, indirect=True)
def test_lazy_charges_at_binades_equal_literal_spans(dev):
    """The same crafted charges with the jumps (and the node batches) on and off (OPT_NOBATCH: every span literally): every
    byte of the record equal after every step, across episode ends."""
    sc = field()
    total = dict(nlazy=0, binade=0, time=0, tie=0, thr_lo=0)
    for i, wu in enumerate(WARM_UPS):
        rows = 8
        w = LazyWitness(MC_THR["threshold"])
        plan = crafted_charges(_offsets(rows), 40 + i)

        def before_step(a, b, k, act):
            live = np.ones(a.B, bool)
            aid = pc._np(a.req.agent_id)
            w.probe(a, live)
            for r, c, e in plan(a, live, aid, act):
                b.mc("ENERGY")[r, c] = e
                w.edited(r, c, e)
        pc.check_batches_equal_event_path(sc, dev, num_envs=rows, steps=30, seed=40 + i, mc=MC_THR, scale2=1.0,
                                          warm_up_time=wu, before_step=before_step)
        for key in total:
            total[key] += w.n[key]
    print("lazy charges, jumps vs literal spans: witnesses", total)
    assert (total["nlazy"] >= 400 and total["binade"] >= 150 and total["time"] >= 20 and total["tie"] >= 10
            and total["thr_lo"] >= 200), total


# ------------------------------------------------------------------ lazy runs cut by the ends of budgeted launches
class CutWitness:
    """launches that end in flight (request -4) with a lazy charge slot whose owed insertion counters grew in that launch: the
    launch's final catch-up cut the run at its own clock, not at an event of the run"""

    def __init__(self):
        self.cs, self.n, self.prev = _pc_cs_fire(), 0, None

    def __call__(self, env):
        E = env.E
        pi = env.view("proc").view(torch.int32)
        lazy = pi[:, :, E["WRSN_PRI_LAZY"]].cpu().numpy() != 0
        cs = pi[:, :, E["WRSN_PRI_PC"]].cpu().numpy() == self.cs
        owed = pc._np(env.view("proc")[:, :, E["WRSN_PR_OWED"]])
        inflight = pc._np(env.req.agent_id) == -4
        if self.prev is not None:
            self.n += int((inflight & (lazy & cs & (owed > self.prev)).any(1)).sum())
        self.prev = owed


BUDGETS = (1, 2, 3, 7)
CUT_CASES = ([pytest.param("cpu", M, b, id="cpu-M%d-b%d" % (M, b)) for M in (3, 16) for b in BUDGETS]
             + [pytest.param(GPU, M, b, id="gpu-M%d-b%d" % (M, b), marks=pytest.mark.gpu) for M in (3, 16) for b in BUDGETS])


@pytest.mark.parametrize("dev,M,budget", CUT_CASES, indirect=["dev"])
def test_lazy_runs_cut_by_launch_ends(dev, M, budget):
    """Step budgets of 1, 2, 3 and 7 end nearly every launch inside a step, where every lazy run is brought up to the launch's
    clock (catch_up_many) and resumed by the next launch; long charges (scale2 = 1) with 3 and 16 chargers.  Every request and
    every byte of the record equal the unbudgeted run's."""
    scs = [synthetic(num_nodes=60, num_targets=60, seed=s, num_gateways=2) for s in (7, 8)]
    w = CutWitness()
    n = pc.check_budget_equals_unbudgeted(scs, dev, num_envs=4, calls=4 * M, seed=budget + M, budget=budget, num_agent=M, scale2=1.0,
                                          launch_probe=w)
    print("budget", budget, "chargers", M, "interrupted launches", n, "cut lazy charges", w.n)
    assert n >= 100 and w.n >= 100, (n, w.n)
