"""GPU: the KZG prover on the B200 — every prover golden case through the single and batch entry points, a seeded soak
checked against closed forms and the device's own verifier, linearity, in-domain proofs, degenerate trusted setups that
force doublings, cancellations and infinite bases through the MSM, mixed batches, n = 0 / 1 / MAX + 1, and the prover
handlers of the conformance-vector runner."""
import ctypes
import json
import random
from pathlib import Path

import numpy as np
import pytest

from oracle import bls_oracle as bo
from oracle import kzg_oracle as ko
from tests import spec_vectors as sv
from tests import spec_vectors_kzg_prover as svp
from tests.golden import make_kzg_golden as mk
from tests.golden import make_kzg_prover_golden as mkp

pytestmark = pytest.mark.gpu
GOLDEN_DIR = Path(__file__).parent / "golden"
SETUP_TEXT = mk.setup_json()
GOLDEN = json.loads((GOLDEN_DIR / "kzg_prover_cases.json").read_text())
TAU_G1 = bo.g1_uncompress(bytes.fromhex(mk.TAU_G1))[1]
R = ko.R


@pytest.fixture(scope="module")
def kzg(engine):
    from ethereum_consensus_b200 import kzg
    return kzg


@pytest.fixture(scope="module")
def lib(engine):
    from ethereum_consensus_b200 import _lib
    return _lib.lib()


@pytest.fixture(scope="module")
def settings(kzg):
    return kzg.kzg_settings_from_json(SETUP_TEXT)


def _code_of(kzg, fn, *a):
    try:
        return 0, fn(*a)
    except kzg.InvalidProof:
        return 5, None
    except kzg.CKzgError:
        return 17, None


def _pt(k: int) -> bytes:
    return bo.g1_compress(ko.to_aff(ko.g1_mul(bo.G1_GEN, k)))


def _add(*cs: bytes) -> bytes:
    pts = [bo.pt_from_affine(ko.F1, bo.g1_uncompress(c)[1]) for c in cs]
    return bo.g1_compress(ko.to_aff(ko.g1_add(*pts)))


def _random_blob(rng) -> bytes:
    return b"".join(rng.randrange(R).to_bytes(32, "big") for _ in range(4096))


def _poly(blob: bytes):
    return [int.from_bytes(blob[32 * i:32 * i + 32], "big") for i in range(4096)]


def test_golden_commit_cases(kzg, lib, settings):
    cases = GOLDEN["commit_cases"]
    blobs = [mkp.build_blob(c["blob"]) for c in cases]
    out, codes = kzg.blob_to_kzg_commitments(blobs, settings)
    assert codes.tolist() == [c["code"] for c in cases]
    for c, blob, o in zip(cases, blobs, out):
        assert bytes(o).hex() == c["commitment"], c["name"]
        buf = ctypes.create_string_buffer(48)
        assert lib.b200_blob_to_kzg_commitment(settings.handle, blob, buf) == c["code"], c["name"]
        assert buf.raw.hex() == c["commitment"], c["name"]   # zeros for a failed blob
        code, got = _code_of(kzg, kzg.blob_to_kzg_commitment, blob, settings)
        assert code == c["code"], c["name"]
        if code == 0:
            assert got.hex() == c["commitment"], c["name"]


def test_golden_point_cases(kzg, settings):
    for c in GOLDEN["point_cases"]:
        code, got = _code_of(kzg, kzg.compute_kzg_proof, mkp.build_blob(c["blob"]), bytes.fromhex(c["z"]), settings)
        assert code == c["code"], c["name"]
        if code == 0:
            assert got == kzg.ProofAndEvaluation(bytes.fromhex(c["proof"]), bytes.fromhex(c["y"])), c["name"]


def test_golden_blob_cases(kzg, settings):
    cases = GOLDEN["blob_cases"]
    blobs = [mkp.build_blob(c["blob"]) for c in cases]
    cs = [bytes.fromhex(c["commitment"]) for c in cases]
    out, codes = kzg.compute_blob_kzg_proofs(blobs, cs, settings)
    assert codes.tolist() == [c["code"] for c in cases]
    for c, blob, cm, o in zip(cases, blobs, cs, out):
        assert bytes(o).hex() == c["proof"], c["name"]
        code, got = _code_of(kzg, kzg.compute_blob_kzg_proof, blob, cm, settings)
        assert code == c["code"], c["name"]
        if code == 0:
            assert got.hex() == c["proof"], c["name"]


def test_seeded_soak(kzg, settings):
    """256 blobs: degree-1 blobs against their closed forms, full random blobs against the device's verifier."""
    rng = random.Random(20261017)
    n_deg1, n_full = 64, 192
    blobs, want_c, want_p = [], [], []
    for _ in range(n_deg1):
        a, b = rng.randrange(R), rng.randrange(R)
        blob, c, p = ko.degree1_case(a, b, TAU_G1)
        blobs.append(blob)
        want_c.append(c)
        want_p.append(p)
    blobs += [_random_blob(rng) for _ in range(n_full)]
    flat = np.frombuffer(b"".join(blobs), np.uint8)
    cs, codes = kzg.blob_to_kzg_commitments(flat, settings)
    assert not codes.any()
    assert [bytes(c) for c in cs[:n_deg1]] == want_c
    ps, codes = kzg.compute_blob_kzg_proofs(flat, np.ascontiguousarray(cs).reshape(-1), settings)
    assert not codes.any()
    assert [bytes(p) for p in ps[:n_deg1]] == want_p
    got = kzg.verify_blob_kzg_proofs(flat, np.ascontiguousarray(cs).reshape(-1), np.ascontiguousarray(ps).reshape(-1), settings)
    assert got.tolist() == [0] * len(blobs)
    mutated = bytearray(blobs[n_deg1 + 3])
    mutated[32 * 100 + 31] ^= 1
    assert kzg.verify_blob_kzg_proofs([bytes(mutated)], [bytes(cs[n_deg1 + 3])], [bytes(ps[n_deg1 + 3])], settings).tolist() == [5]


def test_linearity(kzg, settings):
    rng = random.Random(11)
    a, b = _random_blob(rng), _random_blob(rng)
    s = b"".join(((x + y) % R).to_bytes(32, "big") for x, y in zip(_poly(a), _poly(b)))
    ca, cb, cs = (kzg.blob_to_kzg_commitment(x, settings) for x in (a, b, s))
    assert _add(ca, cb) == cs


def test_compute_kzg_proof_verifies(kzg, settings):
    rng = random.Random(12)
    blob = _random_blob(rng)
    c = kzg.blob_to_kzg_commitment(blob, settings)
    poly = _poly(blob)
    for z in [rng.randrange(R), ko.ROOTS_BRP[5], ko.ROOTS_BRP[4000], 0]:
        zb = z.to_bytes(32, "big")
        r = kzg.compute_kzg_proof(blob, zb, settings)
        assert int.from_bytes(r.evaluation, "big") == ko.evaluate_polynomial_in_evaluation_form(poly, z)
        kzg.verify_kzg_proof(c, zb, r.evaluation, r.proof, settings)
        bad_y = ((int.from_bytes(r.evaluation, "big") + 1) % R).to_bytes(32, "big")
        with pytest.raises(kzg.InvalidProof):
            kzg.verify_kzg_proof(c, zb, bad_y, r.proof, settings)


@pytest.mark.parametrize("kind", ["all_g1", "alternating", "with_infinity"])
def test_degenerate_setups(kzg, kind):
    """Every base G1, -G1 or infinity: commitments are [sum +-f_i]G1, one scalar multiplication in Python each."""
    d = json.loads(SETUP_TEXT)
    g, ng, inf = _pt(1), _pt(R - 1), ko.G1_INFINITY
    if kind == "all_g1":
        pts, sign = [g] * 4096, lambda j: 1
    elif kind == "alternating":
        pts, sign = [g if j % 2 == 0 else ng for j in range(4096)], lambda j: 1 if j % 2 == 0 else -1
    else:
        pts, sign = [inf if j % 3 == 0 else (g if j % 3 == 1 else ng) for j in range(4096)], lambda j: [0, 1, -1][j % 3]
    st = kzg.KzgSettings.load_trusted_setup(pts, [bytes.fromhex(h[2:]) for h in d["g2_monomial"]])
    rng = random.Random(["all_g1", "alternating", "with_infinity"].index(kind))
    blobs = [_random_blob(rng) for _ in range(3)]
    blobs.append(((R - 1).to_bytes(32, "big")) * 4096)        # every term the largest scalar: equal points meet in every sum
    blobs.append(((1 << 254) - 1).to_bytes(32, "big") * 4096)  # long runs of 1-bits: the recoding carry in every window
    blobs.append(rng.randrange(R).to_bytes(32, "big") * 4096)
    out, codes = kzg.blob_to_kzg_commitments(blobs, st)
    assert not codes.any()
    for blob, o in zip(blobs, out):
        poly = _poly(blob)
        k = sum(sign(ko.reverse_bits(i)) * f for i, f in enumerate(poly)) % R
        assert bytes(o) == (_pt(k) if k else ko.G1_INFINITY)


def test_mixed_batches(kzg, settings):
    rng = random.Random(13)
    good = [_random_blob(rng) for _ in range(3)]
    bad = bytearray(good[1])
    bad[32 * 9:32 * 10] = R.to_bytes(32, "big")
    blobs = [good[0], bytes(bad), good[2]]
    out, codes = kzg.blob_to_kzg_commitments(blobs, settings)
    assert codes.tolist() == [0, 17, 0]
    assert bytes(out[1]) == bytes(48)
    single = [kzg.blob_to_kzg_commitment(b, settings) for b in (good[0], good[2])]
    assert [bytes(out[0]), bytes(out[2])] == single
    cs = [single[0], single[0], mk.off_subgroup_point(), single[1]]
    pblobs = [good[0], bytes(bad), good[1], good[2]]
    ps, codes = kzg.compute_blob_kzg_proofs(pblobs, cs, settings)
    assert codes.tolist() == [0, 17, 17, 0]
    assert bytes(ps[1]) == bytes(ps[2]) == bytes(48)
    assert [bytes(ps[0]), bytes(ps[3])] == [kzg.compute_blob_kzg_proof(good[0], single[0], settings),
                                            kzg.compute_blob_kzg_proof(good[2], single[1], settings)]


def test_n0_n1_and_limit(kzg, lib, settings):
    from ethereum_consensus_b200 import _lib
    empty = np.zeros(0, np.uint8)
    out, codes = kzg.blob_to_kzg_commitments(empty, settings)
    assert out.shape == (0, 48) and codes.tolist() == []
    out, codes = kzg.compute_blob_kzg_proofs(empty, empty, settings)
    assert out.shape == (0, 48) and codes.tolist() == []
    assert lib.b200_blob_to_kzg_commitments(settings.handle, None, 0, None, None) == 0
    assert lib.b200_compute_blob_kzg_proofs(settings.handle, None, None, 0, None, None) == 0
    c = GOLDEN["commit_cases"][0]
    out, codes = kzg.blob_to_kzg_commitments([mkp.build_blob(c["blob"])], settings)
    assert codes.tolist() == [0] and bytes(out[0]).hex() == c["commitment"]
    n = kzg.MAX_BLOBS_PER_CALL + 1
    assert lib.b200_blob_to_kzg_commitments(settings.handle, None, n, None, None) == _lib.ERR_BAD_ARG
    assert lib.b200_compute_blob_kzg_proofs(settings.handle, None, None, n, None, None) == _lib.ERR_BAD_ARG


def test_runner_on_synthetic_tree_device(settings, tmp_path):
    base = svp.synthetic_prover_tree(tmp_path / "consensus-spec-tests", GOLDEN, mkp.build_blob)
    impl = svp.DeviceKzgProverImpl(settings)
    n = 0
    for config, fork, handler, case in sv.walk(base, "kzg", svp.KZG_PROVER_HANDLERS):
        passed, detail = svp.run_kzg_prover_case(handler, case, impl)
        assert passed, (handler, case.name, detail)
        n += 1
    assert n == len(GOLDEN["commit_cases"]) + len(GOLDEN["point_cases"]) + len(GOLDEN["blob_cases"]) + 3


@pytest.mark.skipif(sv.vectors_root() is None, reason="consensus-spec-tests not present (offline); set CONSENSUS_SPEC_TESTS")
def test_real_vectors_device(settings):
    impl = svp.DeviceKzgProverImpl(settings)
    n = 0
    for config, fork, handler, case in sv.walk(sv.vectors_root(), "kzg", svp.KZG_PROVER_HANDLERS):
        passed, detail = svp.run_kzg_prover_case(handler, case, impl)
        assert passed, (config, fork, handler, case.name, detail)
        n += 1
    assert n > 0
