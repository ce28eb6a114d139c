"""Known-answer tests of ``oracle/shims/simpy`` (TEST INFRASTRUCTURE: the event kernel under which the unmodified reference
is run to produce the golden fixtures) against what SimPy 4.0.1 (``requirements.txt:52``, not installable here) PUBLISHES:

* the worked examples of its documentation with their printed outputs (README clock example, "Basic Concepts" car
  example, "Process Interaction" sub-process return value, "Events" condition example);
* the scheduling contract the reference leans on (SURVEY §8c): heap key (time, priority, insertion id), URGENT for
  ``Initialize`` and for a numeric ``until``, FIFO among equal keys, ``run(until=processed_event)`` returning at once.

This narrows, but does not close, the "parity unpinned" gap below the golden fixtures: it checks the shim against SimPy's
published behaviour, not against a SimPy wheel."""
import importlib.util
import os
import sys

import pytest

from oracle.ref_runner import reference_root
from tests.helpers import REPO


@pytest.fixture(scope="module")
def simpy():
    path = os.path.join(REPO, "oracle", "shims", "simpy", "__init__.py")
    spec = importlib.util.spec_from_file_location("_shim_simpy", path, submodule_search_locations=[os.path.dirname(path)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules["_shim_simpy"] = mod
    spec.loader.exec_module(mod)
    yield mod
    sys.modules.pop("_shim_simpy", None)


def test_readme_clock_example(simpy):
    """SimPy README: fast 0 / slow 0 / fast 0.5 / slow 1 / fast 1.0 / fast 1.5 — equal times in scheduling order, and
    run(until=2) stops BEFORE the events of t = 2."""
    out = []

    def clock(env, name, tick):
        while True:
            out.append((name, env.now))
            yield env.timeout(tick)

    env = simpy.Environment()
    env.process(clock(env, "fast", 0.5))
    env.process(clock(env, "slow", 1))
    env.run(until=2)
    assert out == [("fast", 0), ("slow", 0), ("fast", 0.5), ("slow", 1), ("fast", 1.0), ("fast", 1.5)]
    assert env.now == 2


def test_basic_concepts_car_example(simpy):
    """'SimPy in 10 Minutes / Basic Concepts': parking 5, driving 2, until=15."""
    out = []

    def car(env):
        while True:
            out.append("Start parking at %d" % env.now)
            yield env.timeout(5)
            out.append("Start driving at %d" % env.now)
            yield env.timeout(2)

    env = simpy.Environment()
    env.process(car(env))
    env.run(until=15)
    assert out == ["Start parking at 0", "Start driving at 5", "Start parking at 7", "Start driving at 12", "Start parking at 14"]


def test_process_return_value_and_run_until_event(simpy):
    """'Events' guide: a process is an event; its return value is the value of `yield process` and of run(until=process)."""
    def sub(env):
        yield env.timeout(1)
        return 23

    def parent(env):
        ret = yield env.process(sub(env))
        return ret

    env = simpy.Environment()
    assert env.run(env.process(parent(env))) == 23
    assert env.now == 1


def test_condition_example(simpy):
    """'Events' guide, condition events: `t1 | t2` fires with the first, `t1 & t2` with the last, `(e1 | e2) & e3`."""
    seen = []

    def proc(env):
        t1, t2 = env.timeout(1, value="spam"), env.timeout(2, value="eggs")
        yield t1 | t2
        seen.append(("or", env.now, t1.processed, t2.processed))
        t1, t2 = env.timeout(1, value="spam"), env.timeout(2, value="eggs")
        yield t1 & t2
        seen.append(("and", env.now, t1.processed, t2.processed))
        e1, e2, e3 = [env.timeout(i) for i in range(3)]
        yield (e1 | e2) & e3
        seen.append(("mix", env.now, all(e.processed for e in (e1, e2, e3))))

    env = simpy.Environment()
    env.process(proc(env))
    env.run()
    assert seen == [("or", 1, True, False), ("and", 3, True, True), ("mix", 5, True)]


def test_run_until_rules(simpy):
    """'Environments' guide: run(until=t) needs t > now; run() ends when the schedule is empty; peek() is the next time."""
    env = simpy.Environment(initial_time=3)
    with pytest.raises(ValueError):
        env.run(until=3)
    env.timeout(4)
    assert env.peek() == 7
    env.run()
    assert env.now == 7 and env.peek() == float("inf")


def test_scheduling_contract(simpy):
    """What the reference depends on (SURVEY §8c), from SimPy 4.0.1 core.py / events.py:
    * a new process starts through an URGENT Initialize event: at one instant it runs before NORMAL events queued earlier;
    * a numeric `until` is an URGENT stop event: no NORMAL event of that instant is processed;
    * equal (time, priority): insertion order;
    * a process that yields an already processed event continues at once, without a trip through the heap;
    * run(until=event that is already processed) returns immediately."""
    order = []
    env = simpy.Environment()

    def late(env, tag):
        order.append(("start", tag, env.now))
        yield env.timeout(0)
        order.append(("after0", tag, env.now))

    def spawner(env):
        yield env.timeout(1)
        t = env.timeout(0)                                   # NORMAL, queued first
        t.callbacks.append(lambda e: order.append(("timeout0", env.now)))
        env.process(late(env, "p"))                          # URGENT Initialize, queued second
        yield env.timeout(0)
        order.append(("spawner", env.now))

    env.process(spawner(env))
    env.run(until=2)
    assert order == [("start", "p", 1), ("timeout0", 1), ("spawner", 1), ("after0", "p", 1)]

    env = simpy.Environment()
    hits = []
    ev = env.timeout(5)
    ev.callbacks.append(lambda e: hits.append(env.now))
    env.run(until=5)
    assert hits == [] and env.now == 5                       # the stop event precedes the NORMAL event of t = 5
    env.run(until=6)
    assert hits == [5]

    env = simpy.Environment()
    done = env.timeout(1)
    env.run(until=2)
    trace = []

    def waiter(env):
        yield done                                           # processed long ago: resume immediately
        trace.append(env.now)
        yield env.timeout(1)
        trace.append(env.now)

    p = env.process(waiter(env))
    assert env.run(until=done) is None and env.now == 2      # already processed: returns at once
    env.run(until=p)
    assert trace == [2, 3]


def _genuine_simpy():
    """A real SimPy distribution (not oracle/shims)?"""
    import importlib.util as iu
    spec = iu.find_spec("simpy")
    if spec is None or not spec.origin:
        return False
    return not os.path.abspath(spec.origin).startswith(os.path.join(REPO, "oracle", "shims"))


@pytest.mark.skipif(not _genuine_simpy(), reason="no genuine simpy distribution in this image (requirements.txt:52 pins simpy==4.0.1)")
@pytest.mark.skipif(reference_root() is None, reason="needs a checkout of the reference (set WRSN_REFERENCE_ROOT)")
def test_goldens_under_genuine_simpy(tmp_path):
    """Pins the one layer the fixtures inherit from the shim: regenerate one pure-network trace and one episode with the
    UNMODIFIED reference under the GENUINE simpy package and demand the committed fixtures byte for byte.  Skipped where no
    simpy wheel exists (this image): until it has run, the SimPy layer of every parity claim is 'unpinned against a wheel'."""
    import subprocess
    env = dict(os.environ, WRSN_REAL_SIMPY="1", WRSN_GOLDEN_OUT=str(tmp_path))
    subprocess.run([sys.executable, os.path.join(REPO, "oracle", "gen_golden.py"), "net:hanoi1000n50", "ep:edge_n50"], check=True, env=env,
                   cwd=REPO, timeout=1800)
    for name in ("net_hanoi1000n50", "ep_edge_n50"):
        new = np.load(os.path.join(str(tmp_path), name + ".npz"), allow_pickle=False)
        old = np.load(os.path.join(REPO, "tests", "golden", name + ".npz"), allow_pickle=False)
        assert sorted(new.files) == sorted(old.files)
        for k in old.files:
            if k.startswith("meta_") or k in ("wall_seconds",):
                continue
            assert np.array_equal(new[k], old[k], equal_nan=True) if old[k].dtype.kind == "f" else np.array_equal(new[k], old[k]), (name, k)
