"""TEST INFRASTRUCTURE ONLY -- run the reference's own hot-path source, unmodified, in this image.

``import pulsarbat`` fails here (astropy, dask and baseband are not installable: no network, not
in the wheelhouse).  The hot-path modules, however, use those packages only for unit bookkeeping
and ``isinstance`` checks, so this loader

* puts the stand-ins of ``oracle/ref_shim`` (astropy.units / astropy.time / dask names) on
  ``sys.modules`` -- ONLY inside ``load()`` and only when the real packages are absent,
* creates an empty ``pulsarbat`` package whose ``__path__`` is ``/root/reference/pulsarbat`` and
  imports from it, WHERE THEY LIE, the files on the path: ``core.py``, ``fft.py``, ``utils.py``,
  ``transforms/`` (``dedispersion.py``, ``transforms.py``) and ``contrib/misc.py`` -- the same
  star-imports the reference's ``__init__.py:9-21`` does, minus ``readers`` (needs ``baseband``)
  and ``pulsar``, of which ``load_predictor()`` imports ``pulsar/predictor.py`` alone (its
  ``phase.py`` needs astropy's Angle machinery; the predictor only hands ``pb.Phase`` the two
  parts it computed, so a two-field record stands in).

Nothing is copied; the reference is read, never written.  Used by oracle/make_ref_golden.py to
freeze reference outputs into tests/golden/ref_golden.npz, and by ``bench.py --impl reference``;
the tests compare with the frozen vectors only."""

import importlib
import os
import sys
import types

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SHIM = os.path.join(_HERE, "ref_shim")


def _has_ref(root):
    return bool(root) and os.path.isfile(
        os.path.join(root, "pulsarbat", "transforms", "dedispersion.py"))


# where the reference's package directory lives: the read-only checkout in the build container,
# else the unmodified pip install under baseline/_ref (git-ignored; it travels to the GPU box,
# where /root/reference does not exist -- __graft_entry__.build() creates it)
REF_ROOT = next((r for r in (os.environ.get("PBK_REFERENCE_ROOT"), "/root/reference",
                             os.path.join(os.path.dirname(_HERE), "baseline", "_ref"))
                 if _has_ref(r)), "/root/reference")


def available():
    return _has_ref(REF_ROOT)


def load():
    """Return (pb, u, Time): the reference package (hot-path subset) and the unit/time modules
    it was imported against."""
    if not available():
        raise RuntimeError(f"reference sources not found under {REF_ROOT}")
    if "pulsarbat" in sys.modules and getattr(sys.modules["pulsarbat"], "_pbk_ref", False):
        pb = sys.modules["pulsarbat"]
        return pb, sys.modules["astropy.units"], sys.modules["astropy.time"].Time
    try:
        import astropy.units  # noqa: F401  (a real astropy wins if it ever appears)
        import dask.array  # noqa: F401
    except ImportError:
        sys.path.insert(0, _SHIM)
        for name in [m for m in sys.modules if m.split(".")[0] in ("astropy", "dask")]:
            del sys.modules[name]
        importlib.import_module("astropy.units")
        importlib.import_module("astropy.time")
        importlib.import_module("dask.array")
        sys.path.remove(_SHIM)

    pb = types.ModuleType("pulsarbat")
    pb.__path__ = [os.path.join(REF_ROOT, "pulsarbat")]
    pb.__file__ = os.path.join(REF_ROOT, "pulsarbat", "__init__.py")
    pb._pbk_ref = True
    sys.modules["pulsarbat"] = pb
    dont = sys.dont_write_bytecode
    sys.dont_write_bytecode = True          # never write __pycache__ into /root/reference
    try:
        for sub, star in (("core", True), ("fft", False), ("utils", False)):
            mod = importlib.import_module(f"pulsarbat.{sub}")
            setattr(pb, sub, mod)
            if star:
                for k in mod.__all__:
                    setattr(pb, k, getattr(mod, k))
        # transforms/__init__.py:5-9 star-imports transforms.py and dedispersion.py
        tr = importlib.import_module("pulsarbat.transforms")
        pb.transforms = tr
        for k in tr.__all__:
            setattr(pb, k, getattr(tr, k))
        # contrib/__init__.py pulls in more than misc.py; bind misc.py alone
        contrib = types.ModuleType("pulsarbat.contrib")
        contrib.__path__ = [os.path.join(REF_ROOT, "pulsarbat", "contrib")]
        sys.modules["pulsarbat.contrib"] = contrib
        misc = importlib.import_module("pulsarbat.contrib.misc")
        contrib.misc, contrib.stft, contrib.istft = misc, misc.stft, misc.istft
        pb.contrib = contrib
    finally:
        sys.dont_write_bytecode = dont
    return pb, sys.modules["astropy.units"], sys.modules["astropy.time"].Time


class _PhaseStub:
    """What pulsar/predictor.py hands to ``pb.Phase``: (integer cycles, fractional cycles).  The
    reference's Phase class (pulsar/phase.py) needs astropy's Angle machinery and is not loaded;
    the predictor only constructs it from the two parts it has computed."""

    def __init__(self, phase1, phase2=0.0):
        self.phase1 = np.asarray(phase1)
        self.phase2 = np.asarray(phase2, dtype=np.float64)


def load_predictor():
    """Return (PhasePredictor, PolycoEntry, u, Time): the reference's pulsar/predictor.py executed
    where it lies, against the astropy stand-ins (QTable, array-capable Time) and with ``pb.Phase``
    replaced by a two-field record."""
    pb, u, Time = load()
    if hasattr(pb, "PhasePredictor"):
        return pb.PhasePredictor, pb.PolycoEntry, u, Time
    if "astropy.table" not in sys.modules:
        sys.path.insert(0, _SHIM)
        try:
            importlib.import_module("astropy.table")
        finally:
            sys.path.remove(_SHIM)
    pb.Phase = _PhaseStub
    pulsar = types.ModuleType("pulsarbat.pulsar")
    pulsar.__path__ = [os.path.join(REF_ROOT, "pulsarbat", "pulsar")]
    sys.modules["pulsarbat.pulsar"] = pulsar
    dont = sys.dont_write_bytecode
    sys.dont_write_bytecode = True
    try:
        pred = importlib.import_module("pulsarbat.pulsar.predictor")
    finally:
        sys.dont_write_bytecode = dont
    pulsar.predictor = pred
    pb.pulsar = pulsar
    pb.PhasePredictor, pb.PolycoEntry = pred.PhasePredictor, pred.PolycoEntry
    return pb.PhasePredictor, pb.PolycoEntry, u, Time
