"""TEST INFRASTRUCTURE ONLY -- never imported by the product path.

Harness that lets the *unmodified* reference (morl-baselines @ a8acdbb, mounted read-only at
/root/reference) be imported in the build container, where its third-party dependencies
(gymnasium, mo_gymnasium, pymoo, cvxpy, pycddlib, matplotlib, seaborn) are not installed.

It registers empty stand-in modules in ``sys.modules`` carrying only the *names* the reference
touches at import time (SURVEY.md Appendix B), and offers a ``FakeEnv`` exposing the attributes
``MOAgent.extract_env_info`` reads (reference ``morl_baselines/common/morl_algorithm.py:248-273``).

Only the golden-data generators under ``tests/golden/`` and ``bench.py`` (its CPU arm, when the
reference is present) may use this module; the tests compare against the stored golden data and
never import the reference.  Without the reference, ``reference_available()`` is False.
"""

from __future__ import annotations

import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("MORL_REFERENCE_ROOT", "/root/reference")


def reference_available() -> bool:
    return os.path.isdir(os.path.join(REFERENCE_ROOT, "morl_baselines"))


from morl_baselines_b200.testing import Box, Discrete, FakeEnv, MultiBinary, _Spec  # noqa: E402,F401  (spaces-only environment shell, shared with bench.py)


# ----------------------------------------------------------------------------------------------
# sys.modules stubs
# ----------------------------------------------------------------------------------------------
def _mod(name, **attrs):
    m = sys.modules.get(name)
    if m is None:
        m = types.ModuleType(name)
        m.__dict__["__graft_stub__"] = True
        sys.modules[name] = m
    for k, v in attrs.items():
        setattr(m, k, v)
    return m


def _have(name):
    try:
        __import__(name)
        return True
    except Exception:
        return False


def install_stubs():
    """Register stand-ins for the reference's missing third-party imports (idempotent)."""
    if not _have("gymnasium"):

        class Env:  # gymnasium.Env
            pass

        class Wrapper:
            def __init__(self, env):
                self.env = env

        spaces = _mod("gymnasium.spaces", Discrete=Discrete, Box=Box, MultiBinary=MultiBinary)
        core = _mod("gymnasium.core", Env=Env)
        wr = _mod("gymnasium.wrappers", RecordVideo=object)
        wr_rec = _mod("gymnasium.wrappers.record_episode_statistics", RecordEpisodeStatistics=object)
        _mod("gymnasium", spaces=spaces, Env=Env, core=core, Wrapper=Wrapper, wrappers=wr, make=None)
        del wr_rec
    if not _have("mo_gymnasium"):
        vec = _mod("mo_gymnasium.wrappers.vector", MOSyncVectorEnv=type("MOSyncVectorEnv", (), {}),
                   MORecordEpisodeStatistics=object)
        wrp = _mod("mo_gymnasium.wrappers", MONormalizeReward=object, MORecordEpisodeStatistics=object, vector=vec)
        _mod("mo_gymnasium", wrappers=wrp, make=None, MORecordEpisodeStatistics=object)
        _mod("mo_gymnasium.utils", MOSyncVectorEnv=type("MOSyncVectorEnv", (), {}))
    if not _have("pymoo"):
        _mod("pymoo")
        _mod("pymoo.util")
        _mod("pymoo.util.ref_dirs", get_reference_directions=_riesz_unavailable)
        _mod("pymoo.indicators")
        _mod("pymoo.indicators.hv", HV=_HVStub)
        _mod("pymoo.indicators.igd", IGD=_IGDStub)
        _mod("pymoo.decomposition")
        _mod("pymoo.decomposition.tchebicheff", Tchebicheff=object)
    if not _have("cvxpy"):
        _mod("cvxpy", SolverError=type("SolverError", (Exception,), {}))
    if not _have("cdd"):
        _mod("cdd")
    if not _have("matplotlib"):
        _mod("matplotlib.pyplot")
        _mod("matplotlib", pyplot=sys.modules["matplotlib.pyplot"])
    if not _have("seaborn"):
        _mod("seaborn")
    if not _have("fire"):
        _mod("fire")


def _riesz_unavailable(*a, **k):
    raise RuntimeError("pymoo is not installed: Riesz-energy reference directions unavailable (parity unpinned, SURVEY 8(c))")


class _HVStub:
    """pymoo.indicators.hv.HV stand-in backed by the in-repo exact hypervolume (minimisation form)."""

    def __init__(self, ref_point):
        self.ref_point = np.asarray(ref_point, dtype=np.float64)

    def __call__(self, points):
        from oracle.hv_oracle import hypervolume_min

        return hypervolume_min(np.asarray(points, dtype=np.float64), self.ref_point)


class _IGDStub:
    def __init__(self, ref_front):
        self.ref = np.asarray(ref_front, dtype=np.float64)

    def __call__(self, points):
        pts = np.asarray(points, dtype=np.float64)
        d = np.linalg.norm(self.ref[:, None, :] - pts[None, :, :], axis=-1)
        return float(d.min(axis=1).mean())


_IMPORTED = {}


def import_reference(modname: str):
    """Import ``morl_baselines.<...>`` from the read-only mount with the stubs installed."""
    if not reference_available():
        raise RuntimeError(f"reference not mounted at {REFERENCE_ROOT}")
    if modname in _IMPORTED:
        return _IMPORTED[modname]
    install_stubs()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    import importlib

    m = importlib.import_module(modname)
    _IMPORTED[modname] = m
    return m
