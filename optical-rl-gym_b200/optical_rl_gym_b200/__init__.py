"""B200-native batched Optical RL-Gym step path (RWA / RMSA / DeepRMSA / RMCSA)."""
from .topology import (TopologyTables, get_topology, load_reference_pickle, nsfnet, read_sndlib_topology,  # noqa: F401
                       read_txt_file, synthetic_ring_chords)

_LAZY = {"OpticalVecEnv": "vec_env", "make": "vec_env", "StepInfo": "vec_env", "COUNTER_NAMES": "vec_env",
         "PolicyRollout": "vec_env"}


def __getattr__(name):      # torch / CUDA are imported lazily so that the topology tools work anywhere
    if name in _LAZY:
        import importlib

        return getattr(importlib.import_module("." + _LAZY[name], __name__), name)
    raise AttributeError(name)
