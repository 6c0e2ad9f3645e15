"""Pulsar timing helpers on the fold path (reference: pulsarbat/pulsar/)."""

from .folding import dedisperse_fold, fold  # noqa: F401
from .predictor import PhasePredictor, PolycoEntry  # noqa: F401
from .search import SinglePulseCandidates, single_pulse_search  # noqa: F401

__all__ = ["PolycoEntry", "PhasePredictor", "fold", "dedisperse_fold", "single_pulse_search",
           "SinglePulseCandidates"]
