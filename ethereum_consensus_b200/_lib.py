"""ctypes binding of the C ABI declared in include/b200_consensus.h.

The CUDA library is the product: there is NO CPU fallback.  `load()` raises if the shared object is missing,
`init()` raises if no B200 is visible.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("B200_LIB", PKG / "libb200_consensus.so"))  # B200_LIB: alternate build for A/B tuning

# return codes (include/b200_consensus.h)
SUCCESS, BAD_ENCODING, POINT_NOT_ON_CURVE, POINT_NOT_IN_GROUP = 0, 1, 2, 3
AGGR_TYPE_MISMATCH, VERIFY_FAIL, PK_IS_INFINITY, BAD_SCALAR = 4, 5, 6, 7
EMPTY_AGGREGATE = 16
KZG_BAD_ARGS = 17
STATE_TRANSITION_INVALID = 18
ERR_CUDA, ERR_NO_DEVICE, ERR_BAD_ARG, ERR_SSZ_MALFORMED, ERR_NOT_INITIALIZED, ERR_LIMIT, ERR_COMM = 0x100, 0x101, 0x102, 0x103, 0x104, 0x105, 0x106
PRESET = {"mainnet": 0, "minimal": 1}

_u8p = C.POINTER(C.c_uint8)
_lib = None
_inited_device = None


class EngineError(RuntimeError):
    """CUDA / argument / SSZ-layout failure reported by the engine (codes >= 0x100)."""

    def __init__(self, code: int, where: str):
        self.code = code
        msg = ""
        if _lib is not None:
            msg = _lib.b200_last_error().decode(errors="replace")
        super().__init__(f"{where}: engine error 0x{code:x} {msg}")


_PROTOS = {
    "b200_init": (C.c_int32, [C.c_int32]),
    "b200_shutdown": (None, []),
    "b200_last_error": (C.c_char_p, []),
    "b200_launch_count": (C.c_uint64, []),
    "b200_last_kernel_ms": (C.c_float, []),
    "b200_sha256": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200_merkleize": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p]),
    "b200_mix_in_length": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_void_p]),
    "b200_is_valid_merkle_branch": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p, C.POINTER(C.c_int32)]),
    "b200_htr_validators": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p]),
    "b200_htr_packed": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint64, C.c_int32, C.c_uint64, C.c_void_p]),
    "b200_htr_beacon_state_deneb": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p]),
    "b200_state_upload_deneb": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(C.c_void_p)]),
    "b200_state_root": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "b200_state_free": (None, [C.c_void_p]),
    "b200_state_update_elements": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200_state_update_bytes": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_size_t]),
    "b200_state_root_incremental": (C.c_int32, [C.c_void_p, C.c_void_p]),
    "b200_htr_beacon_state_deneb_shard": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "b200_htr_beacon_state_deneb_combine": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "b200_compute_shuffled_indices": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_void_p]),
    "b200_get_active_validator_indices": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_uint64, C.c_void_p, C.POINTER(C.c_size_t)]),
    "b200_state_process_epoch_deneb": (C.c_int32, [C.c_void_p, C.c_uint32]),
    "b200_state_process_slots_deneb": (C.c_int32, [C.c_void_p, C.c_uint64]),
    "b200_state_serialized_len": (C.c_int32, [C.c_void_p, C.POINTER(C.c_size_t)]),
    "b200_state_download_deneb": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "b200_state_shuffled_active_indices": (C.c_int32, [C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.c_void_p, C.POINTER(C.c_size_t)]),
    # multi-GPU (comm.cu): the exchange step lives inside the library
    "b200_comm_unique_id": (C.c_int32, [C.c_void_p]),
    "b200_comm_init": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32]),
    "b200_comm_info": (C.c_int32, [C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "b200_comm_destroy": (None, []),
    "b200_collective_count": (C.c_uint64, []),
    "b200_comm_all_gather_bytes": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200_htr_beacon_state_deneb_sharded": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, C.c_void_p]),
    "b200_state_upload_deneb_sharded": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_int32, C.POINTER(C.c_void_p)]),
    "b200_fast_aggregate_verify_batch_sharded": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200_fast_aggregate_verify_batch_mixed": (C.c_int32, [C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "b200_tune": (C.c_int32, [C.c_char_p, C.c_int64]),
    "b200_vm_load_programs": (C.c_int32, [C.c_void_p, C.c_size_t]),
}


def register_protos(protos: dict) -> None:
    _PROTOS.update(protos)
    if _lib is not None:
        _bind(_lib, protos)


def _bind(lib, protos) -> None:
    for name, (res, args) in protos.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported: fail loudly
        fn.restype = res
        fn.argtypes = args


def load():
    """dlopen the CUDA library (no device needed)."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU fallback for this package.")
        lib = C.CDLL(str(LIB_PATH))
        _bind(lib, _PROTOS)
        _lib = lib
    return _lib


def init(device: int | None = None):
    """Bind this process to one GPU (one process per GPU).  Raises EngineError when no B200 is usable."""
    global _inited_device
    lib = load()
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if _inited_device is None:
        rc = lib.b200_init(device)
        if rc != SUCCESS:
            raise EngineError(rc, "b200_init")
        _inited_device = device
    return lib


def lib():
    return init()


def ptr(buf) -> int:
    """Address of a bytes / bytearray / memoryview / numpy array / torch tensor / int pointer (no copy).
    The caller must keep `buf` alive for the duration of the call."""
    if isinstance(buf, int):
        return buf
    if hasattr(buf, "data_ptr"):
        return buf.data_ptr()
    if hasattr(buf, "ctypes"):
        return buf.ctypes.data
    import numpy as np
    a = np.frombuffer(buf, dtype=np.uint8)
    return a.ctypes.data if a.size else 0


def check(rc: int, where: str) -> int:
    if rc >= 0x100:
        raise EngineError(rc, where)
    return rc
