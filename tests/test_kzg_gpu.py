"""GPU: KZG blob-proof verification on the B200 against the oracle's codes — every golden case through all four entry
points, a seeded soak of degree-1 mainnet-setup blobs with adversarial ones mixed in, n = 0 / 1, settings-load errors,
and the conformance vectors when CONSENSUS_SPEC_TESTS is set."""
import ctypes
import json
import random
from pathlib import Path

import numpy as np
import pytest

from oracle import bls_oracle as bo
from oracle import kzg_oracle as ko
from tests import spec_vectors as sv
from tests import spec_vectors_kzg as svk
from tests.golden import make_kzg_golden as mk

pytestmark = pytest.mark.gpu
GOLDEN_DIR = Path(__file__).parent / "golden"
SETUP_TEXT = mk.setup_json()
GOLDEN = json.loads((GOLDEN_DIR / "kzg_cases.json").read_text())


@pytest.fixture(scope="module")
def kzg(engine):
    from ethereum_consensus_b200 import kzg
    return kzg


@pytest.fixture(scope="module")
def settings(kzg):
    return kzg.kzg_settings_from_json(SETUP_TEXT)


@pytest.fixture(scope="module")
def blob_cases():
    return [(c, mk.build_blob(c["blob"]), bytes.fromhex(c["commitment"]), bytes.fromhex(c["proof"])) for c in GOLDEN["blob_cases"]]


def _code_of(kzg, fn, *a):
    try:
        fn(*a)
        return 0
    except kzg.InvalidProof:
        return 5
    except kzg.CKzgError:
        return 17


def test_golden_blob_cases_every_entry_point(kzg, settings, blob_cases):
    from ethereum_consensus_b200 import _lib
    lib = _lib.lib()
    want = [c["code"] for c, *_ in blob_cases]
    # the throughput path: all cases in one call
    got = kzg.verify_blob_kzg_proofs([b for _, b, _, _ in blob_cases], [c for *_, c, _ in blob_cases],
                                     [p for *_, p in blob_cases], settings)
    assert got.tolist() == want
    for (case, blob, c, p) in blob_cases:
        assert lib.b200_verify_blob_kzg_proof(settings.handle, blob, c, p) == case["code"], case["name"]
        assert _code_of(kzg, kzg.verify_blob_kzg_proof, blob, c, p, settings) == case["code"], case["name"]
        assert _code_of(kzg, kzg.verify_blob_kzg_proof_batch, [blob], [c], [p], settings) == case["code"], case["name"]


def test_golden_point_cases(kzg, settings):
    for case in GOLDEN["point_cases"]:
        args = [bytes.fromhex(case[k]) for k in ("commitment", "z", "y", "proof")]
        assert _code_of(kzg, kzg.verify_kzg_proof, *args, settings) == case["code"], case["name"]


def test_golden_batch_cases(kzg, settings, blob_cases):
    by = {c["name"]: (b, cm, p) for c, b, cm, p in blob_cases}
    for case in GOLDEN["batch_cases"]:
        ms = [by[m] for m in case["members"]]
        got = _code_of(kzg, kzg.verify_blob_kzg_proof_batch, [m[0] for m in ms], [m[1] for m in ms], [m[2] for m in ms], settings)
        assert got == case["code"], case["name"]


def _soak_inputs(n, seed):
    """n degree-1 blobs on the mainnet setup, ~4 % adversarial; expected codes by construction (a changed element moves
    y = p(z) off the committed line; an element >= r or a proof outside G1 is malformed)."""
    rng = random.Random(seed)
    tau_g1 = bo.g1_uncompress(bytes.fromhex(GOLDEN["tau_g1"]))[1]
    off_g1 = mk.off_subgroup_point()
    blobs, cs, ps, want = bytearray(), bytearray(), bytearray(), []
    for i in range(n):
        a, b = rng.randrange(ko.R), rng.randrange(ko.R)
        blob, c, p = ko.degree1_case(a, b, tau_g1)
        blob, code = bytearray(blob), 0
        kind = rng.randrange(100)
        if kind == 0:
            j = rng.randrange(4096)
            v = (int.from_bytes(blob[32 * j:32 * j + 32], "big") + 1 + rng.randrange(1000)) % ko.R
            blob[32 * j:32 * j + 32] = v.to_bytes(32, "big")
            code = 5
        elif kind == 1:
            j = rng.randrange(4096)
            blob[32 * j:32 * j + 32] = (ko.R + rng.randrange(1000)).to_bytes(32, "big")
            code = 17
        elif kind == 2:
            p, code = off_g1, 17
        elif kind == 3:
            p, code = bo.g1_compress(ko.to_aff(ko.g1_mul(bo.G1_GEN, b + 1))), 5
        blobs += blob
        cs += c
        ps += p
        want.append(code)
    return np.frombuffer(bytes(blobs), np.uint8), np.frombuffer(bytes(cs), np.uint8), np.frombuffer(bytes(ps), np.uint8), want


def test_seeded_degree1_soak(kzg, settings):
    n = 1024
    blobs, cs, ps, want = _soak_inputs(n, 20240313)
    assert 0 < sum(1 for w in want if w) < n // 10
    got = kzg.verify_blob_kzg_proofs(blobs, cs, ps, settings)
    assert got.tolist() == want
    # the whole-batch check: 0 iff every blob is valid, 17 on any malformed input, else 5
    assert _code_of(kzg, kzg.verify_blob_kzg_proof_batch, blobs, cs, ps, settings) == (17 if 17 in want else 5)
    valid = [i for i, w in enumerate(want) if w == 0]
    fails = [i for i, w in enumerate(want) if w == 5]
    B, C, P = blobs.reshape(n, -1), cs.reshape(n, -1), ps.reshape(n, -1)
    sub = lambda idx: (np.ascontiguousarray(B[idx]).reshape(-1), np.ascontiguousarray(C[idx]).reshape(-1),  # noqa: E731
                       np.ascontiguousarray(P[idx]).reshape(-1))
    assert _code_of(kzg, kzg.verify_blob_kzg_proof_batch, *sub(valid), settings) == 0
    assert _code_of(kzg, kzg.verify_blob_kzg_proof_batch, *sub(valid[:50] + fails[:1]), settings) == 5


def test_n0_and_n1(kzg, settings, blob_cases):
    from ethereum_consensus_b200 import _lib
    lib = _lib.lib()
    empty = np.zeros(0, np.uint8)
    assert kzg.verify_blob_kzg_proofs(empty, empty, empty, settings).tolist() == []
    assert kzg.verify_blob_kzg_proof_batch([], [], [], settings) is None
    assert lib.b200_verify_blob_kzg_proof_batch(settings.handle, None, None, None, 0) == 0
    out = np.full(1, -1, np.int32)
    assert lib.b200_verify_blob_kzg_proofs(settings.handle, None, None, None, 0, out.ctypes.data) == 0 and out[0] == -1
    case, blob, c, p = blob_cases[0]
    assert kzg.verify_blob_kzg_proofs([blob], [c], [p], settings).tolist() == [case["code"]]
    with pytest.raises(kzg.CKzgError):
        kzg.verify_blob_kzg_proof_batch([blob], [c], [], settings)
    assert lib.b200_verify_blob_kzg_proofs(settings.handle, None, None, None, kzg.MAX_BLOBS_PER_CALL + 1, out.ctypes.data) == _lib.ERR_BAD_ARG


def test_settings_load_errors(kzg):
    d = json.loads(SETUP_TEXT)
    with pytest.raises(kzg.CKzgError):   # wrong count
        kzg.kzg_settings_from_json(json.dumps({"g1_lagrange": d["g1_lagrange"][:4095], "g2_monomial": d["g2_monomial"]}))
    with pytest.raises(kzg.CKzgError):
        kzg.kzg_settings_from_json(json.dumps({"g1_lagrange": d["g1_lagrange"], "g2_monomial": d["g2_monomial"][:1]}))
    bad = list(d["g1_lagrange"])
    bad[17] = "0x" + bytes([int(bad[17][2:4], 16) & 0x7F]).hex() + bad[17][4:]   # compression bit cleared
    with pytest.raises(kzg.CKzgError):
        kzg.kzg_settings_from_json(json.dumps({"g1_lagrange": bad, "g2_monomial": d["g2_monomial"]}))
    bad = list(d["g1_lagrange"])
    bad[4000] = "0x" + mk.off_subgroup_point().hex()      # on the curve, not in G1
    with pytest.raises(kzg.CKzgError):
        kzg.kzg_settings_from_json(json.dumps({"g1_lagrange": bad, "g2_monomial": d["g2_monomial"]}))
    bad2 = list(d["g2_monomial"])
    bad2[1] = "0x" + ("c0" + "00" * 94 + "01")              # infinity flag with a payload
    with pytest.raises(kzg.CKzgError):
        kzg.kzg_settings_from_json(json.dumps({"g1_lagrange": d["g1_lagrange"], "g2_monomial": bad2}))
    # a good load still works afterwards
    assert kzg.kzg_settings_from_json(SETUP_TEXT).handle


def test_runner_on_synthetic_tree_device(settings, tmp_path):
    base = svk.synthetic_tree(tmp_path / "consensus-spec-tests", GOLDEN, mk.build_blob, max_blob_cases=32)
    impl = svk.DeviceKzgImpl(settings)
    n = 0
    for config, fork, handler, case in sv.walk(base, "kzg", svk.KZG_HANDLERS):
        passed, detail = svk.run_kzg_case(handler, case, impl)
        assert passed, (handler, case.name, detail)
        n += 1
    assert n >= 30


@pytest.mark.skipif(sv.vectors_root() is None, reason="consensus-spec-tests not present (offline); set CONSENSUS_SPEC_TESTS")
def test_real_vectors_device(settings):
    impl = svk.DeviceKzgImpl(settings)
    n = 0
    for config, fork, handler, case in sv.walk(sv.vectors_root(), "kzg", svk.KZG_HANDLERS):
        passed, detail = svk.run_kzg_case(handler, case, impl)
        assert passed, (config, fork, handler, case.name, detail)
        n += 1
    assert n > 0
