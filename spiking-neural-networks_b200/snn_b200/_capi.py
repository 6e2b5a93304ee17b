"""ctypes binding of include/snn_b200.h (the C-ABI shared library libsnn_b200.so).

The library is the product: there is no Python or CPU fallback.  Loading fails loudly when the
shared object is missing, and every handle creation fails with SNN_GPU_GET_DEVICE_FAILURE when no
CUDA device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SNN_B200_LIB: load a tuning variant of the library (make BUILD=... OUT=... EXTRA=...) instead of the default build
LIB_PATH = os.environ.get("SNN_B200_LIB") or os.path.join(os.path.dirname(_HERE), "libsnn_b200.so")

# ---- enums (include/snn_b200.h) ---------------------------------------------------------------
SNN_OK = 0
SNN_GPU_GET_DEVICE_FAILURE = 7
SNN_GRAPH_PRESYNAPTIC_NOT_FOUND = 16
SNN_GRAPH_POSTSYNAPTIC_NOT_FOUND = 17
SNN_GRAPH_POSITION_NOT_FOUND = 18
SNN_GRAPH_DIMENSIONS_DO_NOT_MATCH = 19
SNN_NET_GRAPH_ID_ALREADY_PRESENT = 32
SNN_NET_POSTSYNAPTIC_ID_NOT_FOUND = 33
SNN_NET_PRESYNAPTIC_ID_NOT_FOUND = 34
SNN_NET_ID_NOT_FOUND_IN_LATTICES = 35
SNN_NET_POSTSYNAPTIC_LATTICE_CANNOT_BE_SPIKE_TRAIN = 36
SNN_NET_CANNOT_CONNECT_WITH_REWARD_MODULATED_CONNECTION = 37
SNN_NET_REWARD_MODULATED_CONNECTION_NOT_COMPATIBLE_INTERNALLY = 38
SNN_NET_CONNECT_FUNCTION_MUST_HAVE_NON_REWARD_MODULATED_LATTICE = 39
SNN_INVALID_ARGUMENT = 64
SNN_UNKNOWN_FIELD = 65
SNN_DTYPE_MISMATCH = 66
SNN_SIZE_MISMATCH = 67
SNN_UNSUPPORTED = 68

MODEL_LIF, MODEL_QIF, MODEL_ADLIF, MODEL_ADEX, MODEL_IZH, MODEL_LEAKY_IZH, MODEL_SIMPLE_LIF, MODEL_HH, MODEL_BCM_IZH = range(9)
NT_APPROXIMATE, NT_DESTEXHE, NT_DISCRETE_SPIKE, NT_EXPONENTIAL_DECAY = range(4)
RC_APPROXIMATE, RC_DESTEXHE, RC_EXPONENTIAL_DECAY = range(3)
TRAIN_POISSON, TRAIN_RATE, TRAIN_PRESET = range(3)
REFRACT_DELTA_DIRAC, REFRACT_EXPONENTIAL_DECAY = range(2)
F32, U32, I32 = range(3)
(OPT_ELECTRICAL_SYNAPSE, OPT_CHEMICAL_SYNAPSE, OPT_DO_PLASTICITY, OPT_UPDATE_GRID_HISTORY, OPT_UPDATE_SPIKE_HISTORY,
 OPT_INTERNAL_CLOCK, OPT_PARALLEL, OPT_RNG_SEED, OPT_UPDATE_AVERAGE_HISTORY, OPT_STEPS_PER_GRAPH,
 OPT_UPDATE_EEG_HISTORY, OPT_HALO_TIMEOUT_MS, OPT_GENERAL_PARTITION, OPT_UPDATE_GRAPH_HISTORY,
 OPT_UPDATE_CONNECTING_GRAPH_HISTORY, OPT_UPDATE_SPIKE_EVENTS, OPT_STEP_PATH, OPT_UNIFORM_TILES, OPT_STENCIL_TILES) = range(19)
# OPT_STEP_PATH (read-only): path + STEP_PATH_MULTI * multi of the last run
# OPT_UNIFORM_TILES (read-only): window-kernel tiles of the last run whose neurons share every parameter (read from one tile row)
# OPT_STENCIL_TILES (read-only): window-kernel tiles of the last run that derived their in-edge indices from the stencil
STEP_PATH_NONE, STEP_PATH_GENERAL, STEP_PATH_WIDE, STEP_PATH_WIDE_SPLIT, STEP_PATH_TMA, STEP_PATH_WIN = range(6)
STEP_PATH_MULTI = 16


class StdpStruct(C.Structure):
    _fields_ = [("a_plus", C.c_float), ("a_minus", C.c_float), ("tau_plus", C.c_float), ("tau_minus", C.c_float),
                ("dt", C.c_float)]


class BcmStruct(C.Structure):
    _fields_ = [("decay", C.c_float), ("average_scalar", C.c_float), ("dt", C.c_float)]


class RstdpStruct(C.Structure):
    _fields_ = [(k, C.c_float) for k in ("dopamine", "tau_d", "tau_c", "a_plus", "a_minus", "tau_plus", "tau_minus", "dt")]


class LatticeDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("model", C.c_int32), ("nt_kinetics", C.c_int32),
                ("receptor_kinetics", C.c_int32), ("rows", C.c_uint32), ("cols", C.c_uint32), ("device", C.c_int32),
                ("part_rank", C.c_int32), ("part_world", C.c_int32)]


class NetworkDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("model", C.c_int32), ("nt_kinetics", C.c_int32),
                ("receptor_kinetics", C.c_int32), ("spike_train", C.c_int32), ("refractoriness", C.c_int32),
                ("device", C.c_int32)]


class SnnError(RuntimeError):
    """A non-zero status from the C ABI; `.status` is the snn_status_t code."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[snn status {status}] {message}")
        self.status = status


_P = C.c_void_p
_u64, _u32, _i32, _i64, _f = C.c_uint64, C.c_uint32, C.c_int32, C.c_int64, C.c_float
_pp = C.POINTER(C.c_void_p)

# name -> (argtypes, restype); every symbol declared in include/snn_b200.h must appear here
SIGNATURES = {
    "snn_abi_version": ([], _i32),
    "snn_status_string": ([_i32], C.c_char_p),
    "snn_lattice_last_error": ([_P], C.c_char_p),
    "snn_network_last_error": ([_P], C.c_char_p),
    "snn_device_count": ([C.POINTER(_i32)], _i32),
    "snn_lattice_create": ([C.POINTER(LatticeDesc), _pp], _i32),
    "snn_lattice_destroy": ([_P], _i32),
    "snn_lattice_rows": ([_P, C.POINTER(_u32), C.POINTER(_u32)], _i32),
    "snn_lattice_size": ([_P, C.POINTER(_u64)], _i32),
    "snn_lattice_field_count": ([_P, C.POINTER(_u32)], _i32),
    "snn_lattice_field_info": ([_P, _u32, C.POINTER(C.c_char_p), C.POINTER(_i32), C.POINTER(_u32)], _i32),
    "snn_lattice_set_field": ([_P, C.c_char_p, _P, _u64, _i32], _i32),
    "snn_lattice_fill_field_f32": ([_P, C.c_char_p, _f], _i32),
    "snn_lattice_fill_field_u32": ([_P, C.c_char_p, _u32], _i32),
    "snn_lattice_fill_field_i32": ([_P, C.c_char_p, _i32], _i32),
    "snn_lattice_get_field": ([_P, C.c_char_p, _P, _u64, _i32], _i32),
    "snn_lattice_set_graph_dense": ([_P, _P, _P, _P, _u32], _i32),
    "snn_lattice_set_graph_csr": ([_P, _P, _P, _P, _u64, _u64], _i32),
    "snn_lattice_set_graph_grid": ([_P, _u32, _f], _i32),
    "snn_lattice_graph_nnz": ([_P, C.POINTER(_u64)], _i32),
    "snn_lattice_get_graph_csr": ([_P, _P, _P, _P, _u64, _u64], _i32),
    "snn_lattice_get_graph_dense": ([_P, _P, _P, _u32], _i32),
    "snn_lattice_lookup_weight": ([_P, _u64, _u64, C.POINTER(_f), C.POINTER(_i32)], _i32),
    "snn_lattice_edit_weight": ([_P, _u64, _u64, _i32, _f], _i32),
    "snn_lattice_get_graph_rows": ([_P, _u64, _u64, _P, _P, _P, _u64, C.POINTER(_u64)], _i32),
    "snn_lattice_get_spike_aggregate": ([_P, _P, _u64], _i32),
    "snn_lattice_set_option": ([_P, _i32, _i64], _i32),
    "snn_lattice_get_option": ([_P, _i32, C.POINTER(_i64)], _i32),
    "snn_lattice_set_plasticity": ([_P, C.POINTER(StdpStruct)], _i32),
    "snn_lattice_get_plasticity": ([_P, C.POINTER(StdpStruct)], _i32),
    "snn_lattice_set_dt": ([_P, _f], _i32),
    "snn_lattice_reset_timing": ([_P], _i32),
    "snn_lattice_run": ([_P, _u64], _i32),
    "snn_lattice_run_timed": ([_P, _u64, C.POINTER(_f), C.POINTER(_u64)], _i32),
    "snn_lattice_set_bcm_plasticity": ([_P, _i32, C.POINTER(BcmStruct)], _i32),
    "snn_lattice_set_reward_modulator": ([_P, _i32, _i32, C.POINTER(RstdpStruct)], _i32),
    "snn_lattice_get_reward_modulator": ([_P, C.POINTER(RstdpStruct)], _i32),
    "snn_lattice_run_with_rewards": ([_P, _P, _u64], _i32),
    "snn_lattice_get_connection_traces": ([_P, _P, _P, _P, _u64], _i32),
    "snn_lattice_set_connection_traces": ([_P, _P, _P, _P, _P, _u64], _i32),
    "snn_lattice_history_len": ([_P, C.POINTER(_u64)], _i32),
    "snn_lattice_get_grid_history": ([_P, _P, _u64], _i32),
    "snn_lattice_get_spike_history": ([_P, _P, _u64], _i32),
    "snn_lattice_get_average_history": ([_P, _P, _u64], _i32),
    "snn_lattice_set_eeg_parameters": ([_P, C.c_float, C.c_float, C.c_float], _i32),
    "snn_lattice_get_eeg_history": ([_P, _P, _u64], _i32),
    "snn_lattice_reset_history": ([_P], _i32),
    "snn_lattice_graph_history_len": ([_P, C.POINTER(_u64), C.POINTER(_u64)], _i32),
    "snn_lattice_get_graph_history": ([_P, _P, _u64], _i32),
    "snn_lattice_spike_event_count": ([_P, C.POINTER(_u64), C.POINTER(_u64)], _i32),
    "snn_lattice_get_spike_events": ([_P, _P, _P, _u64], _i32),
    "snn_partition_begin": ([_u32, _i32, _i32], _u32),
    "snn_lattice_ipc_blob_size": ([], _u32),
    "snn_lattice_ipc_export": ([_P, _P], _i32),
    "snn_lattice_ipc_attach": ([_P, _i32, _P], _i32),
    "snn_lattice_attach_local": ([_P, _i32, _P], _i32),
    "snn_lattice_gpart_wants": ([_P, _i32, _P, _u64, C.POINTER(_u64), C.POINTER(_u32)], _i32),
    "snn_lattice_gpart_set_exports": ([_P, _i32, _P, _u64, _u32], _i32),
    "snn_lattice_gpart_attach": ([_P, _i32, _P], _i32),
    "snn_lattice_gpart_attach_local": ([_P, _i32, _P], _i32),
    "snn_network_create": ([C.POINTER(NetworkDesc), _pp], _i32),
    "snn_network_destroy": ([_P], _i32),
    "snn_network_add_lattice": ([_P, _u64, _u32, _u32], _i32),
    "snn_network_add_spike_train_lattice": ([_P, _u64, _u32, _u32], _i32),
    "snn_network_lattice_size": ([_P, _u64, C.POINTER(_u64)], _i32),
    "snn_network_field_count": ([_P, _u64, C.POINTER(_u32)], _i32),
    "snn_network_field_info": ([_P, _u64, _u32, C.POINTER(C.c_char_p), C.POINTER(_i32), C.POINTER(_u32)], _i32),
    "snn_network_set_field": ([_P, _u64, C.c_char_p, _P, _u64, _i32], _i32),
    "snn_network_fill_field_f32": ([_P, _u64, C.c_char_p, _f], _i32),
    "snn_network_fill_field_u32": ([_P, _u64, C.c_char_p, _u32], _i32),
    "snn_network_fill_field_i32": ([_P, _u64, C.c_char_p, _i32], _i32),
    "snn_network_get_field": ([_P, _u64, C.c_char_p, _P, _u64, _i32], _i32),
    "snn_network_set_preset_firing_times": ([_P, _u64, _P, _P, _u64, _u64], _i32),
    "snn_network_connect_dense": ([_P, _u64, _u64, _P, _P, _u64, _u64], _i32),
    "snn_network_connect_csr": ([_P, _u64, _u64, _P, _P, _P, _u64, _u64], _i32),
    "snn_network_connection_nnz": ([_P, _u64, _u64, C.POINTER(_u64)], _i32),
    "snn_network_get_connection_dense": ([_P, _u64, _u64, _P, _P, _u64, _u64], _i32),
    "snn_network_get_connection_csr": ([_P, _u64, _u64, _P, _P, _P, _u64, _u64], _i32),
    "snn_network_lookup_weight": ([_P, _u64, _u64, _u64, _u64, C.POINTER(_f), C.POINTER(_i32)], _i32),
    "snn_network_edit_weight": ([_P, _u64, _u64, _u64, _u64, _i32, _f], _i32),
    "snn_network_get_spike_aggregate": ([_P, _u64, _P, _u64], _i32),
    "snn_network_set_option": ([_P, _i32, _i64], _i32),
    "snn_network_get_option": ([_P, _i32, C.POINTER(_i64)], _i32),
    "snn_network_set_lattice_option": ([_P, _u64, _i32, _i64], _i32),
    "snn_network_get_lattice_option": ([_P, _u64, _i32, C.POINTER(_i64)], _i32),
    "snn_network_set_plasticity": ([_P, _u64, C.POINTER(StdpStruct)], _i32),
    "snn_network_set_dt": ([_P, _f], _i32),
    "snn_network_reset_timing": ([_P], _i32),
    "snn_network_run": ([_P, _u64], _i32),
    "snn_network_add_reward_modulated_lattice": ([_P, _u64, _u32, _u32], _i32),
    "snn_network_set_reward_modulator": ([_P, _u64, _i32, C.POINTER(RstdpStruct)], _i32),
    "snn_network_get_reward_modulator": ([_P, _u64, C.POINTER(_i32), C.POINTER(RstdpStruct)], _i32),
    "snn_network_set_connection_reward_modulated": ([_P, _u64, _u64, _i32], _i32),
    "snn_network_run_with_rewards": ([_P, _P, _u64], _i32),
    "snn_network_get_connection_traces": ([_P, _u64, _u64, _P, _P, _P, _u64], _i32),
    "snn_network_set_connection_traces": ([_P, _u64, _u64, _P, _P, _P, _P, _u64], _i32),
    "snn_network_run_timed": ([_P, _u64, C.POINTER(_f), C.POINTER(_u64)], _i32),
    "snn_network_history_len": ([_P, _u64, C.POINTER(_u64)], _i32),
    "snn_network_get_grid_history": ([_P, _u64, _P, _u64], _i32),
    "snn_network_get_spike_history": ([_P, _u64, _P, _u64], _i32),
    "snn_network_get_average_history": ([_P, _u64, _P, _u64], _i32),
    "snn_network_set_eeg_parameters": ([_P, _u64, C.c_float, C.c_float, C.c_float], _i32),
    "snn_network_get_eeg_history": ([_P, _u64, _P, _u64], _i32),
    "snn_network_reset_history": ([_P], _i32),
    "snn_network_graph_history_len": ([_P, _u64, _u64, C.POINTER(_u64), C.POINTER(_u64)], _i32),
    "snn_network_get_graph_history": ([_P, _u64, _u64, _P, _u64], _i32),
    "snn_network_spike_event_count": ([_P, _u64, C.POINTER(_u64), C.POINTER(_u64)], _i32),
    "snn_network_get_spike_events": ([_P, _u64, _P, _P, _u64], _i32),
}

_lib = None


def load_library(path: str | None = None) -> C.CDLL:
    """Load libsnn_b200.so and attach the prototypes.  Raises OSError if the extension is not built."""
    global _lib
    if _lib is not None and path is None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise OSError(f"{p} not found: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()' "
                      f"or make -C spiking-neural-networks_b200). There is no CPU fallback.")
    lib = C.CDLL(p)
    for name, (args, res) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.argtypes = args
        fn.restype = res
    if lib.snn_abi_version() != 1:
        raise OSError("libsnn_b200.so ABI version mismatch")
    if path is None:
        _lib = lib
    return lib


def check(lib, status: int, handle=None, network: bool = False):
    if status == SNN_OK:
        return
    if handle is not None:
        msg = (lib.snn_network_last_error if network else lib.snn_lattice_last_error)(handle)
    else:
        msg = lib.snn_lattice_last_error(None)
    text = (msg or b"").decode() or lib.snn_status_string(status).decode()
    raise SnnError(status, text)
