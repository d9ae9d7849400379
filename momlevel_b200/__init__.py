"""momlevel_b200 -- B200-native steric sea level behind the momlevel API.

``import momlevel_b200 as momlevel`` gives the hot-path surface of jkrasting/momlevel
(src/momlevel/__init__.py:25-29): ``steric`` / ``thermosteric`` / ``halosteric``,
``eos.wright`` / ``eos.linear``, ``spice.flament``, ``derived.calc_*``,
``reference.setup_reference_state``, ``util.validate_dataset`` and ``test_data``.
All field arithmetic runs in hand-written sm_100a CUDA kernels (libmomlevel_b200.so)
reached through a C ABI; there is no CPU implementation in this package.
"""

from . import core, derived, distributed, dynamic, eos, reference, spice, test_data, util
from .dynamic import inverse_barometer
from .labeled import DataArray, Dataset
from .steric import halosteric, steric, steric_layers, steric_profile, steric_variants, thermosteric

__version__ = "0.1.0"

__all__ = ["core", "derived", "distributed", "dynamic", "inverse_barometer", "eos", "reference", "spice", "test_data", "util", "DataArray", "Dataset",
           "halosteric", "steric", "steric_layers", "steric_profile", "steric_variants", "thermosteric"]
