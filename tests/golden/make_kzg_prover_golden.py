"""Writes tests/golden/kzg_prover_cases.json: KZG prover cases on the mainnet trusted setup with the oracle's outputs
(tests/kzg_prover_oracle.py).  Blobs are stored as make_kzg_golden recipes, plus
  {"const": hex}        every element the same value
  {"unit": [i, hex]}    element i set, every other zero
python tests/golden/make_kzg_prover_golden.py takes about a minute (about 20 MSMs in Python).
"""
from __future__ import annotations

import json
import random
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import bls_oracle as bo  # noqa: E402
from oracle import kzg_oracle as ko  # noqa: E402
from tests import kzg_prover_oracle as kp  # noqa: E402
from tests.golden import make_kzg_golden as mk  # noqa: E402

GOLDEN = Path(__file__).resolve().parent
OUT = GOLDEN / "kzg_prover_cases.json"


def build_blob(recipe: dict) -> bytes:
    if "const" in recipe:
        return bytes.fromhex(recipe["const"]) * ko.FIELD_ELEMENTS_PER_BLOB
    if "unit" in recipe:
        i, h = recipe["unit"]
        blob = bytearray(ko.BYTES_PER_BLOB)
        blob[32 * i:32 * i + 32] = bytes.fromhex(h)
        return bytes(blob)
    return mk.build_blob(recipe)


def main(out: Path = OUT) -> dict:
    setup = json.loads(mk.setup_json())
    g1_lagrange, _ = ko.load_setup(setup)
    verify = json.loads((GOLDEN / "kzg_cases.json").read_text())
    vby = {c["name"]: c for c in verify["blob_cases"]}
    rng = random.Random(7594)
    fe = lambda v: (v % ko.R).to_bytes(32, "big").hex()  # noqa: E731
    hx = lambda b: b.hex()  # noqa: E731

    a, b = rng.randrange(ko.R), rng.randrange(ko.R)
    blobs = {
        "full_0": vby["full_0"]["blob"], "full_1": vby["full_1"]["blob"], "zero": {"zero": True},
        "const": {"const": fe(rng.randrange(ko.R))}, "all_r_minus_1": {"const": fe(ko.R - 1)},
        "all_2_254_minus_1": {"const": ((1 << 254) - 1).to_bytes(32, "big").hex()},
        "deg1": {"deg1": [hex(a), hex(b)]},
        "element_eq_r": dict(vby["full_0"]["blob"], edits={"7": hx(ko.R.to_bytes(32, "big"))}),
    }
    for i in (0, 1, 2048, 4095):
        blobs[f"unit_{i}"] = {"unit": [i, fe(rng.randrange(ko.R))]}

    commit_cases = []
    for name, rec in blobs.items():
        code, c = kp.blob_to_kzg_commitment_code(build_blob(rec), g1_lagrange)
        commit_cases.append({"name": name, "blob": rec, "commitment": hx(c), "code": code})
    cby = {c["name"]: c for c in commit_cases}
    assert cby["full_0"]["commitment"] == vby["full_0"]["commitment"]
    assert cby["full_1"]["commitment"] == vby["full_1"]["commitment"]
    assert cby["zero"]["commitment"] == ko.G1_INFINITY.hex()
    assert cby["all_r_minus_1"]["commitment"] == bo.g1_compress(ko.to_aff(ko.g1_mul(bo.G1_GEN, ko.R - 1))).hex()
    assert cby["element_eq_r"]["code"] == ko.KZG_BAD_ARGS

    point_cases = []
    r_bytes = ko.R.to_bytes(32, "big")
    pts = [("full_random_z", "full_0", fe(rng.randrange(ko.R))), ("full_z_0", "full_0", fe(0)),
           ("full_z_w0", "full_1", fe(ko.ROOTS_BRP[0])), ("full_z_w1", "full_1", fe(ko.ROOTS_BRP[1])),
           ("full_z_w4095", "full_0", fe(ko.ROOTS_BRP[4095])),
           ("deg1_out_of_domain", "deg1", fe(rng.randrange(ko.R))), ("deg1_in_domain", "deg1", fe(ko.ROOTS_BRP[77])),
           ("zero_blob", "zero", fe(rng.randrange(ko.R))), ("const_blob", "const", fe(rng.randrange(ko.R))),
           ("z_eq_r", "deg1", r_bytes.hex()), ("element_eq_r", "element_eq_r", fe(5))]
    for name, bname, z in pts:
        code, proof, y = kp.compute_kzg_proof_code(build_blob(blobs[bname]), bytes.fromhex(z), g1_lagrange)
        point_cases.append({"name": name, "blob": blobs[bname], "z": z, "proof": hx(proof), "y": hx(y), "code": code})
    pby = {c["name"]: c for c in point_cases}
    g1b = bo.g1_compress(ko.to_aff(ko.g1_mul(bo.G1_GEN, b)))
    assert pby["deg1_out_of_domain"]["proof"] == pby["deg1_in_domain"]["proof"] == g1b.hex()
    assert pby["zero_blob"]["proof"] == pby["const_blob"]["proof"] == ko.G1_INFINITY.hex()

    blob_cases = []
    wrong = bytes.fromhex(cby["deg1"]["commitment"])
    x_ge_p = bytearray(bo.P.to_bytes(48, "big"))
    x_ge_p[0] |= 0x80
    cleared = bytearray(bytes.fromhex(vby["full_0"]["commitment"]))
    cleared[0] &= 0x7F
    bl = [("full_0", "full_0", bytes.fromhex(vby["full_0"]["commitment"])),
          ("full_1", "full_1", bytes.fromhex(vby["full_1"]["commitment"])),
          ("wrong_commitment", "full_0", wrong), ("infinity_commitment", "full_1", ko.G1_INFINITY),
          ("commitment_not_in_g1", "full_0", mk.off_subgroup_point()),
          ("commitment_compression_bit_clear", "full_0", bytes(cleared)), ("commitment_x_ge_p", "full_0", bytes(x_ge_p))]
    for name, bname, c in bl:
        code, proof = kp.compute_blob_kzg_proof_code(build_blob(blobs[bname]), c, g1_lagrange)
        blob_cases.append({"name": name, "blob": blobs[bname], "commitment": hx(c), "proof": hx(proof), "code": code})
    bby = {c["name"]: c for c in blob_cases}
    assert bby["full_0"]["proof"] == vby["full_0"]["proof"] and bby["full_1"]["proof"] == vby["full_1"]["proof"]
    assert [bby[k]["code"] for k in ("commitment_not_in_g1", "commitment_compression_bit_clear", "commitment_x_ge_p")] == [17] * 3

    doc = {"commit_cases": commit_cases, "point_cases": point_cases, "blob_cases": blob_cases}
    parts = [f"{json.dumps(k)}: [\n" + ",\n".join(json.dumps(c) for c in doc[k]) + "\n]" for k in doc]
    out.write_text("{" + ",\n".join(parts) + "}\n")   # one case per line
    return doc


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1 else OUT)
