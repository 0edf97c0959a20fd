"""adcensus_b200 -- B200-native AD-Census stereo matching behind the reference's ADCensusStereo API.

The compute path is the hand-written sm_100a CUDA library ``adcensus_b200/lib/libadcensus_b200.so``
(sources in ``adcensus_b200/csrc``), reached through its C ABI (``include/adcensus_b200.h``).
This package is the Python mirror of the reference's interface for that path
(``ADCensusOption`` and ``ADCensusStereo.Initialize / Match / Reset``, reference
``adcensus_types.h:45-75`` and ``ADCensusStereo.h:14-95``).  There is no CPU fallback: importing
works anywhere, but creating an engine without the CUDA library or without a GPU raises.
"""
from .engine import (ADCensusOption, ADCensusStereo, AdcError, AuxOutputs, Engine, STAGE, TAP, lib_path,  # noqa: F401
                     load_library, Invalid_Float)
from .build import build_library  # noqa: F401

__all__ = ["ADCensusOption", "ADCensusStereo", "AdcError", "AuxOutputs", "Engine", "STAGE", "TAP", "lib_path",
           "load_library", "build_library", "Invalid_Float"]
