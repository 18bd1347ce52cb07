"""The prover half of the deneb polynomial-commitments spec in Python big ints, on top of oracle/kzg_oracle.py (whose
functions it reuses unchanged).  Test infrastructure only: the product never imports it.

`compute_kzg_proof` is the full spec, including compute_quotient_eval_within_domain for z on the domain; the `*_code`
wrappers return (code, output bytes) with the codes of include/b200_consensus.h (0, or 17 = Error::CKzg).
"""
from __future__ import annotations

from typing import Sequence, Tuple

from oracle import bls_oracle as bo
from oracle import kzg_oracle as ko

R = ko.R
N = ko.FIELD_ELEMENTS_PER_BLOB


def brp_bases(g1_lagrange: Sequence[object]):
    """bit_reversal_permutation(g1_lagrange): blob element i pairs with g1_lagrange[reverse_bits(i)]."""
    return [g1_lagrange[ko.reverse_bits(i)] for i in range(N)]


def commit_poly(poly: Sequence[int], g1_lagrange: Sequence[object]) -> bytes:
    return bo.g1_compress(ko.g1_lincomb(brp_bases(g1_lagrange), poly))


def compute_quotient_eval_within_domain(z: int, poly: Sequence[int], y: int) -> int:
    acc = 0
    for f, w in zip(poly, ko.ROOTS_BRP):
        if w == z:
            continue
        acc = (acc + (f - y) * w % R * pow(z * (z - w) % R, -1, R)) % R
    return acc


def quotient(poly: Sequence[int], z: int, y: int):
    q = []
    for f, w in zip(poly, ko.ROOTS_BRP):
        if w == z:
            q.append(compute_quotient_eval_within_domain(z, poly, y))
        else:
            q.append((f - y) * pow(w - z, -1, R) % R)
    return q


def compute_kzg_proof_impl(poly: Sequence[int], z: int, g1_lagrange) -> Tuple[bytes, int]:
    y = ko.evaluate_polynomial_in_evaluation_form(poly, z)
    return commit_poly(quotient(poly, z, y), g1_lagrange), y


def compute_kzg_proof(blob: bytes, z_bytes: bytes, g1_lagrange) -> Tuple[bytes, bytes]:
    """(proof, y as 32 big-endian bytes); raises ko.BadArgs."""
    poly = ko.blob_to_polynomial(blob)
    z = ko.bytes_to_bls_field(z_bytes)
    proof, y = compute_kzg_proof_impl(poly, z, g1_lagrange)
    return proof, y.to_bytes(32, "big")


def compute_blob_kzg_proof(blob: bytes, commitment: bytes, g1_lagrange) -> bytes:
    """The spec's compute_blob_kzg_proof: any valid G1 commitment (not checked against the blob); raises ko.BadArgs."""
    ko.bytes_to_g1(commitment)
    poly = ko.blob_to_polynomial(blob)
    return compute_kzg_proof_impl(poly, ko.compute_challenge(blob, commitment), g1_lagrange)[0]


def blob_to_kzg_commitment_code(blob: bytes, g1_lagrange) -> Tuple[int, bytes]:
    try:
        return ko.OK, commit_poly(ko.blob_to_polynomial(blob), g1_lagrange)
    except ko.BadArgs:
        return ko.KZG_BAD_ARGS, bytes(48)


def compute_kzg_proof_code(blob: bytes, z_bytes: bytes, g1_lagrange) -> Tuple[int, bytes, bytes]:
    try:
        return (ko.OK, *compute_kzg_proof(blob, z_bytes, g1_lagrange))
    except ko.BadArgs:
        return ko.KZG_BAD_ARGS, bytes(48), bytes(32)


def compute_blob_kzg_proof_code(blob: bytes, commitment: bytes, g1_lagrange) -> Tuple[int, bytes]:
    try:
        return ko.OK, compute_blob_kzg_proof(blob, commitment, g1_lagrange)
    except ko.BadArgs:
        return ko.KZG_BAD_ARGS, bytes(48)
