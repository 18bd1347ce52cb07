"""CPU: the prover oracle (tests/kzg_prover_oracle.py) — the prover golden file regenerates identically, in- and
out-of-domain proofs pass the oracle's verifier, the closed forms (degree-1, constant, unit blobs) agree with its MSM, and
the prover handlers of the conformance-vector runner pass on a synthetic tree (and on the real vectors when
CONSENSUS_SPEC_TESTS is set)."""
import json
import random
from pathlib import Path

import pytest

from oracle import bls_oracle as bo
from oracle import kzg_oracle as ko
from tests import kzg_prover_oracle as kp
from tests import spec_vectors as sv
from tests import spec_vectors_kzg_prover as svp
from tests.golden import make_kzg_golden as mk
from tests.golden import make_kzg_prover_golden as mkp

GOLDEN_DIR = Path(__file__).parent / "golden"
GOLDEN = json.loads((GOLDEN_DIR / "kzg_prover_cases.json").read_text())
R = ko.R


@pytest.fixture(scope="module")
def setup():
    return json.loads(mk.setup_json())


@pytest.fixture(scope="module")
def g1_lagrange(setup):
    return ko.load_setup(setup)[0]


@pytest.fixture(scope="module")
def tau_g2(setup):
    return ko.load_setup(setup)[1][1]


def _pt(k: int) -> bytes:
    return bo.g1_compress(ko.to_aff(ko.g1_mul(bo.G1_GEN, k)))


def test_golden_regenerates_identically(tmp_path):
    out = tmp_path / "kzg_prover_cases.json"
    mkp.main(out)
    assert out.read_bytes() == (GOLDEN_DIR / "kzg_prover_cases.json").read_bytes()


def test_proofs_verify_in_and_out_of_domain(g1_lagrange, tau_g2):
    rng = random.Random(21)
    blob = b"".join(rng.randrange(R).to_bytes(32, "big") for _ in range(4096))
    c = kp.blob_to_kzg_commitment_code(blob, g1_lagrange)[1]
    for z in (rng.randrange(R), ko.ROOTS_BRP[9]):
        proof, y = kp.compute_kzg_proof(blob, z.to_bytes(32, "big"), g1_lagrange)
        assert ko.verify_kzg_proof(c, z.to_bytes(32, "big"), y, proof, tau_g2) == ko.OK
        y_bad = ((int.from_bytes(y, "big") + 1) % R).to_bytes(32, "big")
        assert ko.verify_kzg_proof(c, z.to_bytes(32, "big"), y_bad, proof, tau_g2) == ko.VERIFY_FAIL


def test_closed_forms(g1_lagrange):
    tau_g1 = bo.g1_uncompress(bytes.fromhex(mk.TAU_G1))[1]
    a, b = 12345, 67890
    blob, c, p = ko.degree1_case(a, b, tau_g1)
    assert kp.blob_to_kzg_commitment_code(blob, g1_lagrange) == (0, c)
    for z in (99, ko.ROOTS_BRP[3]):
        assert kp.compute_kzg_proof(blob, z.to_bytes(32, "big"), g1_lagrange) == (p, ((a + b * z) % R).to_bytes(32, "big"))
    k = 424242
    const = k.to_bytes(32, "big") * 4096
    assert kp.blob_to_kzg_commitment_code(const, g1_lagrange) == (0, _pt(k))            # P1: the bases sum to G1
    assert kp.compute_kzg_proof(const, (5).to_bytes(32, "big"), g1_lagrange)[0] == ko.G1_INFINITY
    for i in (0, 1, 2048, 4095):
        unit = mkp.build_blob({"unit": [i, (7).to_bytes(32, "big").hex()]})
        want = bo.g1_compress(ko.to_aff(ko.g1_mul(g1_lagrange[ko.reverse_bits(i)], 7)))
        assert kp.blob_to_kzg_commitment_code(unit, g1_lagrange) == (0, want), i


def test_golden_closed_forms():
    by = {c["name"]: c for c in GOLDEN["commit_cases"]}
    k = int(by["const"]["blob"]["const"], 16)
    assert by["const"]["commitment"] == _pt(k).hex()
    assert by["all_2_254_minus_1"]["commitment"] == _pt((1 << 254) - 1).hex()
    a, b = (int(v, 16) for v in by["deg1"]["blob"]["deg1"])
    tau_g1 = bo.g1_uncompress(bytes.fromhex(mk.TAU_G1))[1]
    assert by["deg1"]["commitment"] == ko.degree1_case(a, b, tau_g1)[1].hex()


def test_runner_on_synthetic_tree_oracle(setup, tmp_path):
    # the cheap cases only: the oracle runs one Python MSM (seconds) per valid case
    names = {"zero", "element_eq_r", "unit_0", "unit_4095", "zero_blob", "const_blob", "z_eq_r", "commitment_not_in_g1",
             "commitment_x_ge_p", "commitment_compression_bit_clear"}
    base = svp.synthetic_prover_tree(tmp_path / "consensus-spec-tests", GOLDEN, mkp.build_blob, names=names)
    impl = svp.OracleKzgProverImpl(setup)
    n = 0
    for config, fork, handler, case in sv.walk(base, "kzg", svp.KZG_PROVER_HANDLERS):
        passed, detail = svp.run_kzg_prover_case(handler, case, impl)
        assert passed, (handler, case.name, detail)
        n += 1
    assert n == sum(c["name"] in names for k in ("commit_cases", "point_cases", "blob_cases") for c in GOLDEN[k]) + 3


@pytest.mark.skipif(sv.vectors_root() is None, reason="consensus-spec-tests not present (offline); set CONSENSUS_SPEC_TESTS")
def test_real_vectors_oracle(setup):
    impl = svp.OracleKzgProverImpl(setup)
    n = 0
    for config, fork, handler, case in sv.walk(sv.vectors_root(), "kzg", svp.KZG_PROVER_HANDLERS):
        passed, detail = svp.run_kzg_prover_case(handler, case, impl)
        assert passed, (config, fork, handler, case.name, detail)
        n += 1
    assert n > 0
