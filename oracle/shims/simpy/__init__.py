"""SimPy-4.0.1-semantics shim (TEST INFRASTRUCTURE, oracle side only).

The reference pins ``simpy==4.0.1`` (requirements.txt:52) but
SimPy is not installed in this image and there is no network.  This module
restates the part of SimPy's published scheduling contract that the reference
uses (call sites: NetworkIO.py:33; WRSN.py:43,53,62,127,302,307-311;
Network.py:72-78; Node.py:57,65; BaseStation.py:31; MobileCharger.py:44-132):

* heap key ``(now + delay, priority, eid)``; ``eid`` is a global schedule counter;
* ``Timeout`` / ``Event.succeed`` / process completion are NORMAL (1);
  ``Initialize`` (process start) and a numeric ``until`` are URGENT (0);
* ``step()`` detaches ``callbacks`` (sets it to ``None``) before calling them;
* ``Process._resume`` keeps driving the generator while the yielded event has
  already been processed (``callbacks is None``);
* ``Condition`` (``&`` / ``|``) checks already-processed operands at
  construction, succeeds at ``now`` with NORMAL priority, and on being
  processed removes its ``_check`` callbacks from its operands, recursively for
  nested conditions;
* ``run(until=event)`` returns immediately if the event is already processed.

Only the product's tests, ``__graft_entry__.smoke`` and ``bench.py``'s CPU
baseline may import this.  It was written from the published SimPy 4.0.1
behaviour, not checked against a SimPy wheel (none available): the SimPy layer
of the oracle is therefore "parity unpinned" against real SimPy, while
everything above it is the unmodified reference source.
"""
from heapq import heappush, heappop
from itertools import count

__version__ = "4.0.1-shim"

URGENT = 0
NORMAL = 1
PENDING = object()


class StopSimulation(Exception):
    @classmethod
    def callback(cls, event):
        if event._ok:
            raise cls(event._value)
        raise event._value


class EmptySchedule(Exception):
    pass


class Event:
    def __init__(self, env):
        self.env = env
        self.callbacks = []
        self._value = PENDING
        self._ok = None

    @property
    def triggered(self):
        return self._value is not PENDING

    @property
    def processed(self):
        return self.callbacks is None

    @property
    def ok(self):
        return self._ok

    @property
    def value(self):
        if self._value is PENDING:
            raise AttributeError("value of %r is not yet available" % self)
        return self._value

    def succeed(self, value=None):
        if self._value is not PENDING:
            raise RuntimeError("%r has already been triggered" % self)
        self._ok = True
        self._value = value
        self.env.schedule(self)
        return self

    def fail(self, exception):
        if self._value is not PENDING:
            raise RuntimeError("%r has already been triggered" % self)
        self._ok = False
        self._value = exception
        self.env.schedule(self)
        return self

    def __and__(self, other):
        return Condition(self.env, Condition.all_events, [self, other])

    def __or__(self, other):
        return Condition(self.env, Condition.any_events, [self, other])


class Timeout(Event):
    def __init__(self, env, delay, value=None):
        if delay < 0:
            raise ValueError("Negative delay %s" % delay)
        self.env = env
        self.callbacks = []
        self._value = value
        self._delay = delay
        self._ok = True
        env.schedule(self, NORMAL, delay)


class Initialize(Event):
    def __init__(self, env, process):
        self.env = env
        self.callbacks = [process._resume]
        self._value = None
        self._ok = True
        env.schedule(self, URGENT)


class Process(Event):
    def __init__(self, env, generator):
        if not hasattr(generator, "throw"):
            raise ValueError("%s is not a generator." % generator)
        self.env = env
        self.callbacks = []
        self._value = PENDING
        self._ok = None
        self._generator = generator
        self._target = Initialize(env, self)

    @property
    def is_alive(self):
        return self._value is PENDING

    def _resume(self, event):
        self.env._active_proc = self
        while True:
            try:
                if event._ok:
                    event = self._generator.send(event._value)
                else:
                    event._defused = True
                    exc = event._value
                    event = self._generator.throw(type(exc), exc)
            except StopIteration as e:
                event = None
                self._ok = True
                self._value = e.args[0] if len(e.args) else None
                self.env.schedule(self)
                break
            except BaseException as e:
                event = None
                self._ok = False
                self._value = e
                self.env.schedule(self)
                break
            try:
                if event.callbacks is not None:
                    event.callbacks.append(self._resume)
                    break
            except AttributeError:
                raise RuntimeError("Invalid yield value %r" % (event,))
        self._target = event
        self.env._active_proc = None


class ConditionValue:
    def __init__(self):
        self.events = []


class Condition(Event):
    def __init__(self, env, evaluate, events):
        super().__init__(env)
        self._evaluate = evaluate
        self._events = tuple(events)
        self._count = 0
        if not self._events:
            self.succeed(ConditionValue())
            return
        for event in self._events:
            if self.env != event.env:
                raise ValueError("It is not allowed to mix events from different environments")
        for event in self._events:
            if event.callbacks is None:
                self._check(event)
            else:
                event.callbacks.append(self._check)
        self.callbacks.append(self._build_value)

    def _populate_value(self, value):
        for event in self._events:
            if isinstance(event, Condition):
                event._populate_value(value)
            elif event.callbacks is None:
                value.events.append(event)

    def _build_value(self, event):
        self._remove_check_callbacks()
        if event._ok:
            self._value = ConditionValue()
            self._populate_value(self._value)

    def _remove_check_callbacks(self):
        for event in self._events:
            if event.callbacks and self._check in event.callbacks:
                event.callbacks.remove(self._check)
            if isinstance(event, Condition):
                event._remove_check_callbacks()

    def _check(self, event):
        if self._value is not PENDING:
            return
        self._count += 1
        if not event._ok:
            event._defused = True
            self.fail(event._value)
        elif self._evaluate(self._events, self._count):
            self.succeed()

    @staticmethod
    def all_events(events, count):
        return len(events) == count

    @staticmethod
    def any_events(events, count):
        return count > 0 or len(events) == 0


class AllOf(Condition):
    def __init__(self, env, events):
        super().__init__(env, Condition.all_events, events)


class AnyOf(Condition):
    def __init__(self, env, events):
        super().__init__(env, Condition.any_events, events)


class Environment:
    def __init__(self, initial_time=0):
        self._now = initial_time
        self._queue = []
        self._eid = count()
        self._active_proc = None
        # test hook (not part of SimPy): called as trace(now, priority, eid, event)
        self._trace = None

    @property
    def now(self):
        return self._now

    @property
    def active_process(self):
        return self._active_proc

    def process(self, generator):
        return Process(self, generator)

    def timeout(self, delay=0, value=None):
        return Timeout(self, delay, value)

    def event(self):
        return Event(self)

    def all_of(self, events):
        return AllOf(self, events)

    def any_of(self, events):
        return AnyOf(self, events)

    def schedule(self, event, priority=NORMAL, delay=0):
        heappush(self._queue, (self._now + delay, priority, next(self._eid), event))

    def peek(self):
        try:
            return self._queue[0][0]
        except IndexError:
            return float("inf")

    def step(self):
        try:
            self._now, prio, eid, event = heappop(self._queue)
        except IndexError:
            raise EmptySchedule()
        if self._trace is not None:
            self._trace(self._now, prio, eid, event)
        callbacks, event.callbacks = event.callbacks, None
        for callback in callbacks:
            callback(event)
        if not event._ok and not hasattr(event, "_defused"):
            exc = type(event._value)(*event._value.args)
            exc.__cause__ = event._value
            raise exc

    def run(self, until=None):
        if until is not None:
            if not isinstance(until, Event):
                at = float(until)
                if at <= self.now:
                    raise ValueError("until(=%s) must be > the current simulation time." % at)
                until = Event(self)
                until._ok = True
                until._value = None
                self.schedule(until, URGENT, at - self.now)
            elif until.callbacks is None:
                return until.value
            until.callbacks.append(StopSimulation.callback)
        try:
            while True:
                self.step()
        except StopSimulation as exc:
            return exc.args[0]
        except EmptySchedule:
            if until is not None:
                assert not until.triggered
                raise RuntimeError('No scheduled events left but "until" event was not triggered: %s' % until)
        return None
