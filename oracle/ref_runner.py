"""Run the UNMODIFIED reference (a checkout of the original project) under the oracle shims.

TEST INFRASTRUCTURE.  Used only (a) here, in the build container, to generate the
golden fixtures under ``tests/golden/`` (see ``oracle/gen_golden.py``) and to
validate the C restatement ``oracle/wrsn_oracle.c``; (b) by ``tools/time_python_reference.py``,
which times the unmodified Python reference on the host cores of the build container
(``profiles/r02_python_reference.jsonl``).  ``bench.py --impl reference`` does NOT use this
file: the reference's sources do not exist on the GPU box, its CPU arm is the C restatement.
Nothing in the product package imports this file.

``WRSN_REAL_SIMPY=1``: when a genuine ``simpy`` distribution is importable, use it instead of
``oracle/shims/simpy`` (tests/test_simpy_shim.py::test_goldens_under_genuine_simpy regenerates
fixtures under it; no such wheel exists in this image, so that test is skipped here).

The reference root is looked up in this order: ``$WRSN_REFERENCE_ROOT``,
``<repo>/baseline/_ref``.
"""
import os
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
_REPO = os.path.dirname(_HERE)


def reference_root():
    for cand in (os.environ.get("WRSN_REFERENCE_ROOT"), os.path.join(_REPO, "baseline", "_ref")):
        if cand and os.path.isfile(os.path.join(cand, "rl_env", "WRSN.py")):
            return cand
    return None


def load_reference():
    """Import the reference modules; returns a namespace with WRSN, NetworkIO, MobileCharger, root."""
    root = reference_root()
    if root is None:
        raise RuntimeError("reference sources not found (set WRSN_REFERENCE_ROOT)")
    shims = os.path.join(_HERE, "shims")
    if os.environ.get("WRSN_REAL_SIMPY") == "1":
        import simpy  # noqa: F401 - the genuine package, imported BEFORE the shim directory gets on sys.path
        if os.path.abspath(os.path.dirname(simpy.__file__)).startswith(os.path.abspath(shims)):
            raise RuntimeError("WRSN_REAL_SIMPY=1 but `simpy` resolves to oracle/shims")
    for p in (shims, root):
        if p not in sys.path:
            sys.path.insert(0, p)
    from rl_env.WRSN import WRSN  # noqa: E402
    from physical_env.network.NetworkIO import NetworkIO  # noqa: E402
    from physical_env.mc.MobileCharger import MobileCharger  # noqa: E402

    class NS:
        pass
    ns = NS()
    ns.WRSN, ns.NetworkIO, ns.MobileCharger, ns.root = WRSN, NetworkIO, MobileCharger, root
    ns.scenario_dir = os.path.join(root, "physical_env", "network", "network_scenarios")
    ns.mc_type = os.path.join(root, "physical_env", "mc", "mc_types", "default.yaml")
    return ns
