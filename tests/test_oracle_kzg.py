"""CPU: the KZG oracle (oracle/kzg_oracle.py) against identities of the mainnet trusted setup, its own fixture prover and
the committed golden file; the KZG spec-vector runner on a synthetic tree (on the real tree when CONSENSUS_SPEC_TESTS is set)."""
import json
from pathlib import Path

import pytest

from oracle import bls_oracle as bo
from oracle import kzg_oracle as ko
from tests import spec_vectors as sv
from tests import spec_vectors_kzg as svk
from tests.golden import make_kzg_golden as mk

GOLDEN_DIR = Path(__file__).parent / "golden"
SETUP = json.loads(mk.setup_json())
GOLDEN = json.loads((GOLDEN_DIR / "kzg_cases.json").read_text())


@pytest.fixture(scope="module")
def setup_points():
    return ko.load_setup(SETUP)


def test_setup_shape():
    import hashlib
    assert hashlib.sha256(mk.setup_json().encode()).hexdigest() == mk.SETUP_JSON_SHA256   # the reference's file, byte for byte
    assert len(SETUP["g1_lagrange"]) == 4096 and len(SETUP["g2_monomial"]) == 65
    assert bo.g2_uncompress(bytes.fromhex(SETUP["g2_monomial"][0][2:]))[1] == bo.G2_GEN


def test_p1_lagrange_points_sum_to_generator(setup_points):
    g1, _ = setup_points
    assert ko.to_aff(ko.g1_add(*[bo.pt_from_affine(ko.F1, a) for a in g1])) == bo.G1_GEN


def test_p2_tau_g1_by_msm_pairs_with_tau_g2(setup_points):
    g1, g2 = setup_points
    tau_g1 = ko.tau_g1_from_lagrange(g1)
    assert bo.g1_compress(tau_g1).hex() == mk.TAU_G1 == GOLDEN["tau_g1"]
    neg_g1 = bo.G1_GEN_NEG
    assert bo.pairing_check([(tau_g1, bo.G2_GEN), (neg_g1, g2[1])])
    # the bit-reversed reading of the setup does not give [tau]G1
    brp = ko.g1_lincomb([g1[ko.reverse_bits(j)] for j in range(4096)], ko.ROOTS)
    assert not bo.pairing_check([(brp, bo.G2_GEN), (neg_g1, g2[1])])


def test_msm_matches_double_and_add():
    pts = [ko.to_aff(ko.g1_mul(bo.G1_GEN, k)) for k in (3, 5, 7, 11)]
    ks = [ko.R - 1, 2, 1 << 200, 12345]
    want = ko.to_aff(ko.g1_add(*[ko.g1_mul(p, k) for p, k in zip(pts, ks)]))
    assert ko.g1_lincomb(pts, ks) == want


def test_golden_regenerates_identically(tmp_path):
    out = tmp_path / "kzg_cases.json"
    mk.main(out)
    assert out.read_text() == (GOLDEN_DIR / "kzg_cases.json").read_text()


def test_oracle_proofs_verify_and_mutations_fail():
    tau_g1 = bo.g1_uncompress(bytes.fromhex(GOLDEN["tau_g1"]))[1]
    tau_g2 = bo.g2_uncompress(bytes.fromhex(SETUP["g2_monomial"][1][2:]))[1]
    blob, c, p = ko.degree1_case(12345, 678910, tau_g1)
    assert ko.verify_blob_kzg_proof(blob, c, p, tau_g2) == ko.OK
    bad = bytearray(blob)
    bad[31] ^= 1
    assert ko.verify_blob_kzg_proof(bytes(bad), c, p, tau_g2) == ko.VERIFY_FAIL
    z = 99
    y = (12345 + 678910 * z) % ko.R
    assert ko.verify_kzg_proof(c, z.to_bytes(32, "big"), y.to_bytes(32, "big"), p, tau_g2) == ko.OK
    assert ko.verify_kzg_proof(c, z.to_bytes(32, "big"), (y + 1).to_bytes(32, "big"), p, tau_g2) == ko.VERIFY_FAIL
    by = {c["name"]: c["code"] for c in GOLDEN["blob_cases"]}
    assert by["full_0"] == by["full_1"] == 0 and by["swapped_proofs"] == ko.VERIFY_FAIL


def test_kzg_runner_on_synthetic_tree(tmp_path):
    base = svk.synthetic_tree(tmp_path / "consensus-spec-tests", GOLDEN, mk.build_blob)
    impl = svk.OracleKzgImpl(SETUP)
    seen = {}
    for config, fork, handler, case in sv.walk(base, "kzg", svk.KZG_HANDLERS):
        passed, detail = svk.run_kzg_case(handler, case, impl)
        assert passed, (handler, case.name, detail)
        seen[handler] = seen.get(handler, 0) + 1
    assert set(seen) == set(svk.KZG_HANDLERS) and sum(seen.values()) >= 20, seen


REAL = sv.vectors_root()


@pytest.mark.skipif(REAL is None, reason="consensus-spec-tests not present (offline); set CONSENSUS_SPEC_TESTS")
def test_kzg_oracle_against_real_vectors():
    impl = svk.OracleKzgImpl(SETUP)
    n = 0
    for config, fork, handler, case in sv.walk(REAL, "kzg", svk.KZG_HANDLERS):
        passed, detail = svk.run_kzg_case(handler, case, impl)
        assert passed, (config, fork, handler, case.name, detail)
        n += 1
    assert n > 0
