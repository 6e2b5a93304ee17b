"""snn_b200 — reference-shaped Python front end over the B200 C-ABI library (libsnn_b200.so).

The CUDA library is the product; this package holds no compute and no CPU fallback.
"""
from . import _capi
from ._capi import SnnError, load_library
from .backend import CudaLatticeBackend, CudaNetworkBackend
from .lattice import (AverageVoltageHistory, EEGHistory, GraphHistory, GridVoltageHistory, Lattice, LatticeNetwork,
                      RewardModulatedConnection, RewardModulatedLattice, RewardModulatedLatticeNetwork, SpikeEvents,
                      SpikeHistory, SpikeTrainLattice, TraceRSTDP)
from .neurons import *  # noqa: F401,F403
