"""Python big-int restatement of the deneb polynomial-commitments spec (verification side, and a fixture-only prover)
on top of bls_oracle.py.  Test infrastructure only: the product (ethereum_consensus_b200.kzg) never imports it.

Codes follow include/b200_consensus.h: 0 valid, 5 (VERIFY_FAIL) = Error::InvalidProof, 17 (KZG_BAD_ARGS) =
Error::CKzg(..) for any malformed input.

The trusted setup's `g1_lagrange` is in natural order: g1_lagrange[j] = [L_j(tau)]G1 for the Lagrange basis over
w^0, w^1, ... (w = 7^((r-1)/4096)); the spec bit-reverses it where it uses it.  Two identities pin that reading
(tests/test_oracle_kzg.py): sum_j g1_lagrange[j] = G1 (P1) and T = sum_j w^j g1_lagrange[j] = [tau]G1 with
e(T, G2) = e(G1, g2_monomial[1]) (P2).
"""
from __future__ import annotations

import hashlib
from typing import List, Optional, Sequence

from oracle import bls_oracle as bo

R = bo.R
F1 = bo.F1
FIELD_ELEMENTS_PER_BLOB = 4096
BYTES_PER_BLOB = 32 * FIELD_ELEMENTS_PER_BLOB
PRIMITIVE_ROOT_OF_UNITY = 7
FIAT_SHAMIR_PROTOCOL_DOMAIN = b"FSBLOBVERIFY_V1_"
RANDOM_CHALLENGE_KZG_BATCH_DOMAIN = b"RCKZGBATCH___V1_"
OK, VERIFY_FAIL, KZG_BAD_ARGS = 0, 5, 17
G1_INFINITY = bytes([0xC0]) + bytes(47)

OMEGA = pow(PRIMITIVE_ROOT_OF_UNITY, (R - 1) // FIELD_ELEMENTS_PER_BLOB, R)


def reverse_bits(i: int, bits: int = 12) -> int:
    return int(format(i, f"0{bits}b")[::-1], 2)


ROOTS = [pow(OMEGA, i, R) for i in range(FIELD_ELEMENTS_PER_BLOB)]
ROOTS_BRP = [ROOTS[reverse_bits(i)] for i in range(FIELD_ELEMENTS_PER_BLOB)]


class BadArgs(Exception):
    pass


# ---------------------------------------------------------------------------------------------------- decoding
def bytes_to_bls_field(b: bytes) -> int:
    if len(b) != 32:
        raise BadArgs("field element length")
    v = int.from_bytes(b, "big")
    if v >= R:
        raise BadArgs("field element >= r")
    return v


def blob_to_polynomial(blob: bytes) -> List[int]:
    if len(blob) != BYTES_PER_BLOB:
        raise BadArgs("blob length")
    return [bytes_to_bls_field(blob[32 * i:32 * i + 32]) for i in range(FIELD_ELEMENTS_PER_BLOB)]


def bytes_to_g1(b: bytes):
    """validate_kzg_g1: decompress + subgroup check; the infinity encoding is valid (None)."""
    if len(b) != 48:
        raise BadArgs("point length")
    code, a = bo.g1_uncompress(b)
    if code != 0:
        raise BadArgs("point does not decode")
    if a is not None and not bo.in_subgroup(F1, a):
        raise BadArgs("point not in G1")
    return a


def hash_to_bls_field(data: bytes) -> int:
    return int.from_bytes(hashlib.sha256(data).digest(), "big") % R


def compute_challenge(blob: bytes, commitment: bytes) -> int:
    data = FIAT_SHAMIR_PROTOCOL_DOMAIN + FIELD_ELEMENTS_PER_BLOB.to_bytes(16, "big") + blob + commitment
    return hash_to_bls_field(data)


def evaluate_polynomial_in_evaluation_form(poly: Sequence[int], z: int) -> int:
    n = len(poly)
    if z in ROOTS_BRP:
        return poly[ROOTS_BRP.index(z)]
    acc = 0
    for f, w in zip(poly, ROOTS_BRP):
        acc = (acc + f * w * pow(z - w, -1, R)) % R
    return acc * (pow(z, n, R) - 1) * pow(n, -1, R) % R


# ---------------------------------------------------------------------------------------------------- points
def g1_mul(a, k: int):
    return bo.pt_mul(F1, bo.pt_from_affine(F1, a), k % R)


def g1_add(*pts):
    acc = bo.pt_inf(F1)
    for p in pts:
        acc = bo.pt_add(F1, acc, p)
    return acc


def to_aff(p):
    return bo.pt_to_affine(F1, p)


def g1_lincomb(points: Sequence[object], scalars: Sequence[int], window: int = 8):
    """sum_i [s_i] P_i (affine points, None = infinity) by bucket accumulation (Pippenger): ~10x fewer additions than
    4 096 independent double-and-add chains, which keeps the fixture MSMs at seconds in Python."""
    jac = [bo.pt_from_affine(F1, a) for a in points]
    scalars = [s % R for s in scalars]
    total = bo.pt_inf(F1)
    for w in reversed(range((255 + window - 1) // window)):
        for _ in range(window):
            total = bo.pt_double(F1, total)
        buckets = [bo.pt_inf(F1) for _ in range(1 << window)]
        for p, s in zip(jac, scalars):
            d = (s >> (w * window)) & ((1 << window) - 1)
            if d:
                buckets[d] = bo.pt_add(F1, buckets[d], p)
        run, acc = bo.pt_inf(F1), bo.pt_inf(F1)
        for d in range((1 << window) - 1, 0, -1):
            run = bo.pt_add(F1, run, buckets[d])
            acc = bo.pt_add(F1, acc, run)
        total = bo.pt_add(F1, total, acc)
    return to_aff(total)


# ---------------------------------------------------------------------------------------------------- verification
def verify_kzg_proof_impl(commitment, z: int, y: int, proof, tau_g2) -> bool:
    """e(C - [y]G1 + [z]pi, -G2) * e(pi, [tau]G2) == 1  <=>  e(C - [y]G1, G2) == e(pi, [tau - z]G2)."""
    p = to_aff(g1_add(bo.pt_from_affine(F1, commitment), g1_mul(bo.G1_GEN, R - y), g1_mul(proof, z) if proof else bo.pt_inf(F1)))
    neg_g2 = (bo.G2_GEN[0], bo.f2_neg(bo.G2_GEN[1]))
    return bo.pairing_check([(p, neg_g2), (proof, tau_g2)])


def verify_kzg_proof(commitment: bytes, z: bytes, y: bytes, proof: bytes, tau_g2) -> int:
    try:
        c, zz, yy, pi = bytes_to_g1(commitment), bytes_to_bls_field(z), bytes_to_bls_field(y), bytes_to_g1(proof)
    except BadArgs:
        return KZG_BAD_ARGS
    return OK if verify_kzg_proof_impl(c, zz, yy, pi, tau_g2) else VERIFY_FAIL


def blob_inputs(blob: bytes, commitment: bytes, proof: bytes):
    """(C, z, y, pi) of verify_blob_kzg_proof; raises BadArgs."""
    c = bytes_to_g1(commitment)
    poly = blob_to_polynomial(blob)
    z = compute_challenge(blob, commitment)
    y = evaluate_polynomial_in_evaluation_form(poly, z)
    return c, z, y, bytes_to_g1(proof)


def verify_blob_kzg_proof(blob: bytes, commitment: bytes, proof: bytes, tau_g2) -> int:
    try:
        c, z, y, pi = blob_inputs(blob, commitment, proof)
    except BadArgs:
        return KZG_BAD_ARGS
    return OK if verify_kzg_proof_impl(c, z, y, pi, tau_g2) else VERIFY_FAIL


def batch_challenge(commitments: Sequence[bytes], zs, ys, proofs: Sequence[bytes]) -> int:
    data = RANDOM_CHALLENGE_KZG_BATCH_DOMAIN + FIELD_ELEMENTS_PER_BLOB.to_bytes(8, "big") + len(commitments).to_bytes(8, "big")
    for c, z, y, p in zip(commitments, zs, ys, proofs):
        data += c + z.to_bytes(32, "big") + y.to_bytes(32, "big") + p
    return hash_to_bls_field(data)


def verify_blob_kzg_proof_batch(blobs: Sequence[bytes], commitments: Sequence[bytes], proofs: Sequence[bytes], tau_g2) -> int:
    if not len(blobs) == len(commitments) == len(proofs):
        return KZG_BAD_ARGS
    if not blobs:
        return OK
    try:
        ins = [blob_inputs(b, c, p) for b, c, p in zip(blobs, commitments, proofs)]
    except BadArgs:
        return KZG_BAD_ARGS
    cs, zs, ys, pis = zip(*ins)
    r = batch_challenge(commitments, zs, ys, proofs)
    rp = [pow(r, i, R) for i in range(len(blobs))]
    proof_lincomb = g1_add(*[g1_mul(p, s) for p, s in zip(pis, rp) if p])
    terms = [g1_add(bo.pt_from_affine(F1, c), g1_mul(bo.G1_GEN, R - y), g1_mul(p, z) if p else bo.pt_inf(F1))
             for c, z, y, p in zip(cs, zs, ys, pis)]
    rhs = g1_add(*[bo.pt_mul(F1, t, s) for t, s in zip(terms, rp)])
    neg_g2 = (bo.G2_GEN[0], bo.f2_neg(bo.G2_GEN[1]))
    ok = bo.pairing_check([(to_aff(rhs), neg_g2), (to_aff(proof_lincomb), tau_g2)])
    return OK if ok else VERIFY_FAIL


# ---------------------------------------------------------------------------------------------------- fixture prover
def field_bytes(v: int) -> bytes:
    return (v % R).to_bytes(32, "big")


def degree1_case(a: int, b: int, tau_g1):
    """p(X) = a + bX: blob element i = a + b w^brp(i), commitment [a]G1 + [b][tau]G1, proof [b]G1 at any z (p(X) - p(z) =
    b (X - z)).  Valid mainnet-setup triples without an MSM, given T = [tau]G1 (P2)."""
    blob = b"".join(field_bytes(a + b * w) for w in ROOTS_BRP)
    commitment = bo.g1_compress(to_aff(g1_add(g1_mul(bo.G1_GEN, a), g1_mul(tau_g1, b))))
    proof = bo.g1_compress(to_aff(g1_mul(bo.G1_GEN, b)))
    return blob, commitment, proof


def blob_to_kzg_commitment(blob: bytes, g1_lagrange: Sequence[object]) -> bytes:
    """g1_lincomb(bit_reversal_permutation(g1_lagrange), blob_to_polynomial(blob)); `g1_lagrange` as affine points."""
    poly = blob_to_polynomial(blob)
    return bo.g1_compress(g1_lincomb([g1_lagrange[reverse_bits(i)] for i in range(FIELD_ELEMENTS_PER_BLOB)], poly))


def compute_blob_kzg_proof(blob: bytes, commitment: bytes, g1_lagrange: Sequence[object]) -> bytes:
    """The quotient (p(X) - y) / (X - z) in evaluation form, committed; z outside the domain (probability 1 - 2^-243)."""
    poly = blob_to_polynomial(blob)
    z = compute_challenge(blob, commitment)
    assert z not in ROOTS_BRP
    y = evaluate_polynomial_in_evaluation_form(poly, z)
    q = [(f - y) * pow(w - z, -1, R) % R for f, w in zip(poly, ROOTS_BRP)]
    return bo.g1_compress(g1_lincomb([g1_lagrange[reverse_bits(i)] for i in range(FIELD_ELEMENTS_PER_BLOB)], q))


def load_setup(d: dict):
    """(g1_lagrange affine points, g2_monomial affine points) of a parsed trusted_setup JSON."""
    g1 = [bo.g1_uncompress(bytes.fromhex(h[2:]))[1] for h in d["g1_lagrange"]]
    g2 = [bo.g2_uncompress(bytes.fromhex(h[2:]))[1] for h in d["g2_monomial"]]
    return g1, g2


def tau_g1_from_lagrange(g1_lagrange: Sequence[object]):
    """T = sum_j w^j g1_lagrange[j] (natural order) = [tau]G1."""
    return g1_lincomb(list(g1_lagrange), ROOTS)
