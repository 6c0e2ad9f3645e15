"""Transforms on the hot path (reference: pulsarbat/transforms/)."""

from .dedispersion import (DM, DispersionMeasure, coherent_dedispersion,  # noqa: F401
                           dedisperse_detect, dedisperse_trials, incoherent_dedispersion,
                           incoherent_dedispersion_trials, overlap_save_dedispersion)
from .transforms import freq_shift, time_shift  # noqa: F401

__all__ = ["DM", "DispersionMeasure", "coherent_dedispersion", "incoherent_dedispersion",
           "dedisperse_detect", "dedisperse_trials", "incoherent_dedispersion_trials",
           "overlap_save_dedispersion", "time_shift", "freq_shift"]
