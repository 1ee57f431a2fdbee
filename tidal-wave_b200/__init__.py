"""tidal-wave_b200 -- B200-native hot path of arielnetworks/tidal-wave (Farneback flow -> span sampling ->
OK / SUSPICIOUS / ERROR).  The directory name carries a hyphen (the reference's repo name); import it as

    import tidalwave_b200            # alias module at the repo root
    # or: importlib.import_module("tidal-wave_b200")

Contents: csrc/ (sm_100a CUDA kernels + C ABI + dispatcher), api.py (ctypes binding + mirror of the reference's
operator interface), synth.py (seeded synthetic screenshot pairs).
"""
from . import dist, synth, tidalwave  # noqa: F401
from .tidalwave import TidalWave, create, run  # noqa: F401
from .api import (LIB_PATH, MAX_CHANGE_REGIONS, MAX_IGNORE, MAX_INTENSITY_CELLS, imread_gray, OpticalFlow, OpticalFlowParameter, Pool,  # noqa: F401
                  declared_symbols, load, set_default_arithmetic, tw_change_region, tw_flow_param, tw_intensity_cell, tw_rect, tw_result,
                  tw_vector)
