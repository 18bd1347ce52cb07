"""Host-side mirror of the reference's SSZ merkleization surface, backed by the CUDA library.

Mirrors what `ethereum_consensus::ssz::prelude` re-exports from ssz_rs
(/root/reference/ethereum-consensus/src/ssz/mod.rs:4-7): `merkleize`, `mix_in_length`,
`is_valid_merkle_branch`, and `hash_tree_root` for the containers on the hot path
(`deneb::BeaconState`, /root/reference/ethereum-consensus/src/deneb/beacon_state.rs:13-64;
`List<Validator, N>`, /root/reference/ethereum-consensus/src/phase0/validator.rs:10-26).
Every hash is computed on the GPU; there is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
from typing import Sequence

from . import _lib

BYTES_PER_CHUNK = 32


class MerkleizationError(ValueError):
    """Mirrors ssz_rs `MerkleizationError` (surfaced as `Error::Merkleization`, error.rs:16-17)."""


def _out32():
    return (C.c_uint8 * 32)()


def _rc(rc: int, where: str) -> None:
    if rc == _lib.ERR_LIMIT:
        raise MerkleizationError(f"{where}: input exceeds limit")
    if rc == _lib.ERR_SSZ_MALFORMED:
        raise MerkleizationError(f"{where}: malformed SSZ")
    _lib.check(rc, where)


def hash(data) -> bytes:  # noqa: A001 - mirrors crypto::hash (crypto/bls.rs:12-20)
    out = _out32()
    _rc(_lib.lib().b200_sha256(_lib.ptr(data), len(data), out), "hash")
    return bytes(out)


def merkleize(chunks, limit: int | None = None) -> bytes:
    """`merkleize(chunks, limit)`; `chunks` is a bytes-like of n*32 bytes (or a sequence of 32-byte values)."""
    if not isinstance(chunks, (bytes, bytearray, memoryview)) and not hasattr(chunks, "ctypes") and not hasattr(chunks, "data_ptr"):
        chunks = b"".join(bytes(c) for c in chunks)
    nbytes = chunks.nbytes if hasattr(chunks, "nbytes") else len(chunks)
    if nbytes % 32:
        raise MerkleizationError("chunk data is not a multiple of 32 bytes")
    out = _out32()
    _rc(_lib.lib().b200_merkleize(_lib.ptr(chunks), nbytes // 32, limit or 0, out), "merkleize")
    return bytes(out)


def mix_in_length(root: bytes, length: int) -> bytes:
    out = _out32()
    _rc(_lib.lib().b200_mix_in_length(_lib.ptr(root), length, out), "mix_in_length")
    return bytes(out)


def is_valid_merkle_branch(leaf: bytes, branch: Sequence[bytes], depth: int, index: int, root: bytes) -> bool:
    """ssz_rs `is_valid_merkle_branch` (used at phase0/block_processing.rs:428-437, deneb/blob_sidecar.rs:58-63)."""
    if len(branch) < depth:
        return False
    flat = b"".join(bytes(b) for b in branch[:depth])
    ok = C.c_int32(0)
    _rc(_lib.lib().b200_is_valid_merkle_branch(_lib.ptr(leaf), _lib.ptr(flat), depth, index, _lib.ptr(root), C.byref(ok)),
        "is_valid_merkle_branch")
    return bool(ok.value)


def hash_tree_root_validators(ssz, n: int | None = None, limit: int = 1 << 40) -> bytes:
    """hash_tree_root(List<Validator, limit>) from the list's SSZ bytes (n x 121)."""
    nbytes = ssz.nbytes if hasattr(ssz, "nbytes") else len(ssz)
    if n is None:
        if nbytes % 121:
            raise MerkleizationError("validator bytes not a multiple of 121")
        n = nbytes // 121
    out = _out32()
    _rc(_lib.lib().b200_htr_validators(_lib.ptr(ssz), n, limit, out), "hash_tree_root(validators)")
    return bytes(out)


def hash_tree_root_packed(data, limit_chunks: int, is_list: bool, length: int = 0) -> bytes:
    nbytes = data.nbytes if hasattr(data, "nbytes") else len(data)
    out = _out32()
    _rc(_lib.lib().b200_htr_packed(_lib.ptr(data), nbytes, limit_chunks, 1 if is_list else 0, length, out),
        "hash_tree_root(packed)")
    return bytes(out)


def hash_tree_root_beacon_state(ssz, preset: str = "mainnet") -> bytes:
    """`state.hash_tree_root()` for a deneb BeaconState given as SSZ bytes (host memory; pinned is faster)."""
    nbytes = ssz.nbytes if hasattr(ssz, "nbytes") else len(ssz)
    out = _out32()
    _rc(_lib.lib().b200_htr_beacon_state_deneb(_lib.ptr(ssz), nbytes, _lib.PRESET[preset], out),
        "hash_tree_root(BeaconState)")
    return bytes(out)


def _count_validators(ssz, preset: str) -> int:
    """Length of `validators` read from the two offsets in the fixed part (deneb/beacon_state.rs:26-63)."""
    import struct
    hist = 8192 if preset == "mainnet" else 64
    o = 8 + 32 + 8 + 16 + 112 + 2 * 32 * hist + 4 + 72 + 4 + 8   # ... eth1_deposit_index, then the validators offset
    nbytes = ssz.nbytes if hasattr(ssz, "nbytes") else len(ssz)
    if nbytes < o + 8:
        return 0   # malformed: b200_state_upload_deneb reports it
    v_off, b_off = struct.unpack("<II", C.string_at(_lib.ptr(ssz) + o, 8))   # any host buffer (bytes, numpy, pinned tensor)
    return (b_off - v_off) // 121


class DeviceBeaconState:
    """A deneb BeaconState resident in HBM: upload once, `hash_tree_root()` costs kernels only."""

    def __init__(self, ssz, preset: str = "mainnet", sharded: bool = False):
        """`sharded`: the state is spread over the ranks of the library's communicator (parallel.comm_init first; every
        rank constructs it and calls hash_tree_root together; root only)."""
        nbytes = ssz.nbytes if hasattr(ssz, "nbytes") else len(ssz)
        self._h = C.c_void_p()
        self.n_validators = _count_validators(ssz, preset)
        fn = _lib.lib().b200_state_upload_deneb_sharded if sharded else _lib.lib().b200_state_upload_deneb
        _rc(fn(_lib.ptr(ssz), nbytes, _lib.PRESET[preset], C.byref(self._h)), "state_upload")

    def hash_tree_root(self) -> bytes:
        out = _out32()
        _rc(_lib.lib().b200_state_root(self._h, out), "state_root")
        return bytes(out)

    # ---- incremental re-hash (SURVEY.md §8f-2): patch the resident state, then re-hash only the dirty paths ----
    FIELDS = {"validators": (0, 121), "balances": (1, 8), "previous_epoch_participation": (2, 1),
              "current_epoch_participation": (3, 1), "inactivity_scores": (4, 8)}

    def update_elements(self, field: str, indices, values) -> None:
        """Overwrite elements `indices` of one of the five big lists; `values` = their SSZ encodings back to back
        (121-byte Validator records, little-endian u64, or participation-flag bytes)."""
        fid, elem = self.FIELDS[field]
        idx = np.ascontiguousarray(indices, dtype=np.uint64)
        vals = np.frombuffer(values, dtype=np.uint8) if isinstance(values, (bytes, bytearray)) else np.ascontiguousarray(values).view(np.uint8).reshape(-1)
        if vals.size != idx.size * elem:
            raise ValueError(f"{field}: expected {idx.size * elem} value bytes, got {vals.size}")
        _rc(_lib.lib().b200_state_update_elements(self._h, fid, _lib.ptr(idx), _lib.ptr(vals), idx.size), "state_update_elements")

    def update_bytes(self, ssz_offset: int, data) -> None:
        """Overwrite bytes [ssz_offset, ssz_offset+len(data)) of the uploaded serialization (any field, same layout)."""
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        _rc(_lib.lib().b200_state_update_bytes(self._h, ssz_offset, _lib.ptr(buf), buf.size), "state_update_bytes")

    def hash_tree_root_incremental(self) -> bytes:
        out = _out32()
        _rc(_lib.lib().b200_state_root_incremental(self._h, out), "state_root_incremental")
        return bytes(out)

    def to_ssz(self) -> np.ndarray:
        """SSZ serialization of the current resident state (the big lists come back from HBM)."""
        n = C.c_size_t(0)
        _rc(_lib.lib().b200_state_serialized_len(self._h, C.byref(n)), "state_serialized_len")
        out = np.empty(n.value, dtype=np.uint8)
        _rc(_lib.lib().b200_state_download_deneb(self._h, _lib.ptr(out), out.size), "state_download")
        return out

    def close(self) -> None:
        if self._h:
            _lib.lib().b200_state_free(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def shard_roots(ssz, preset: str, rank: int, world: int) -> bytes:
    """This rank's five big-list subtree roots (160 bytes) — see b200_htr_beacon_state_deneb_shard."""
    nbytes = ssz.nbytes if hasattr(ssz, "nbytes") else len(ssz)
    out = (C.c_uint8 * 160)()
    _rc(_lib.lib().b200_htr_beacon_state_deneb_shard(_lib.ptr(ssz), nbytes, _lib.PRESET[preset], rank, world, out),
        "shard_roots")
    return bytes(out)


def combine_roots(ssz, preset: str, world: int, all_roots: bytes) -> bytes:
    nbytes = ssz.nbytes if hasattr(ssz, "nbytes") else len(ssz)
    if world < 1 or len(all_roots) != world * 160:
        raise ValueError(f"all_roots must hold world x 5 x 32 = {world * 160} bytes, got {len(all_roots)}")
    out = _out32()
    _rc(_lib.lib().b200_htr_beacon_state_deneb_combine(_lib.ptr(ssz), nbytes, _lib.PRESET[preset], world,
                                                       _lib.ptr(all_roots), out), "combine_roots")
    return bytes(out)
