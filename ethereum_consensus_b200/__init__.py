"""ethereum_consensus_b200 — B200-native drop-in for the crypto/SSZ hot path of ralexstokes/ethereum_consensus.

`crypto` mirrors `ethereum_consensus::crypto` (BLS), `kzg` its KZG blob-proof verification, `ssz` mirrors the merkleization surface of
`ethereum_consensus::ssz::prelude`; both call the sm_100a CUDA library through the C ABI in
include/b200_consensus.h.  Importing the package does not need a GPU; calling into it does.
"""
from . import _lib  # noqa: F401

__all__ = ["_lib", "ssz", "crypto", "kzg", "state"]
