"""Transforms on the hot path (reference: pulsarbat/transforms/)."""

from .dedispersion import (DM, DispersionMeasure, FDMTTrials,  # noqa: F401
                           coherent_dedispersion, dedisperse_detect, dedisperse_trials,
                           fdmt_dedispersion_trials, incoherent_dedispersion,
                           incoherent_dedispersion_trials, overlap_save_dedispersion)
from .rfi import SpectralKurtosis, sk_thresholds, spectral_kurtosis  # noqa: F401
from .transforms import freq_shift, time_shift  # noqa: F401

__all__ = ["DM", "DispersionMeasure", "coherent_dedispersion", "incoherent_dedispersion",
           "dedisperse_detect", "dedisperse_trials", "incoherent_dedispersion_trials",
           "fdmt_dedispersion_trials", "FDMTTrials", "overlap_save_dedispersion", "time_shift", "freq_shift", "spectral_kurtosis",
           "sk_thresholds", "SpectralKurtosis"]
