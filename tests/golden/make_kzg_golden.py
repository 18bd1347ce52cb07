"""Writes tests/golden/kzg_cases.json: KZG verification cases on the mainnet trusted setup with the oracle's codes.

Blobs are 128 KiB, so the file stores each blob as a recipe that `build_blob` expands:
  {"random": seed}      element i = SHA-256(seed || be32(i)) mod r (full degree; commitment and proof by MSM)
  {"deg1": [a, b]}      p(X) = a + bX (commitment [a]G1 + [b]T, proof [b]G1, T = [tau]G1 from P2; no MSM)
  {"zero": true}        the zero blob (commitment and proof: the infinity encoding)
  "edits": {i: hex}     element i replaced by those 32 bytes afterwards
Every code is computed by oracle/kzg_oracle.py (python tests/golden/make_kzg_golden.py, about a minute).
"""
from __future__ import annotations

import hashlib
import json
import random
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parents[2]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from oracle import bls_oracle as bo  # noqa: E402
from oracle import kzg_oracle as ko  # noqa: E402

GOLDEN = Path(__file__).resolve().parent
# the mainnet trusted setup (the reference's deneb/presets/trusted_setup.json) as raw compressed points: 4 096 x 48 bytes of
# g1_lagrange, then 65 x 96 bytes of g2_monomial.  setup_json() rebuilds that JSON file byte for byte (SHA-256 pinned).
SETUP = GOLDEN / "trusted_setup_4096.bin"
SETUP_JSON_SHA256 = "2ad295c46d027293d3b30dae97962dc4df8dfd988a2f02f6fe818db75f8c2526"
OUT = GOLDEN / "kzg_cases.json"
TAU_G1 = "ad3eb50121139aa34db1d545093ac9374ab7bca2c0f3bf28e27c8dcd8fc7cb42d25926fc0c97b336e9f0fb35e5a04c81"


def setup_points():
    """(g1_lagrange, g2_monomial) as lists of compressed points."""
    raw = SETUP.read_bytes()
    n1 = ko.FIELD_ELEMENTS_PER_BLOB * 48
    return [raw[i:i + 48] for i in range(0, n1, 48)], [raw[i:i + 96] for i in range(n1, len(raw), 96)]


def setup_json() -> str:
    g1, g2 = setup_points()
    return json.dumps({"g1_lagrange": ["0x" + p.hex() for p in g1], "g2_monomial": ["0x" + p.hex() for p in g2]}, indent=2) + "\n"


def build_blob(recipe: dict) -> bytes:
    if "random" in recipe:
        seed = recipe["random"].encode()
        blob = b"".join(ko.field_bytes(int.from_bytes(hashlib.sha256(seed + i.to_bytes(4, "big")).digest(), "big"))
                        for i in range(ko.FIELD_ELEMENTS_PER_BLOB))
    elif "deg1" in recipe:
        a, b = (int(v, 16) for v in recipe["deg1"])
        blob = b"".join(ko.field_bytes(a + b * w) for w in ko.ROOTS_BRP)
    else:
        blob = bytes(ko.BYTES_PER_BLOB)
    blob = bytearray(blob)
    for i, h in recipe.get("edits", {}).items():
        blob[32 * int(i):32 * int(i) + 32] = bytes.fromhex(h)
    return bytes(blob)


def off_subgroup_point() -> bytes:
    """The compressed encoding of the first on-curve point (smallest x) that is not in G1."""
    x = 1
    while True:
        y2 = (x ** 3 + 4) % bo.P
        y = pow(y2, (bo.P + 1) // 4, bo.P)
        if y * y % bo.P == y2 and not bo.in_subgroup(bo.F1, (x, y)):
            return bo.g1_compress((x, y))
        x += 1


def main(out: Path = OUT) -> dict:
    setup = json.loads(setup_json())
    g1_lagrange, g2_monomial = ko.load_setup(setup)
    tau_g2 = g2_monomial[1]
    tau_g1 = ko.tau_g1_from_lagrange(g1_lagrange)
    assert bo.g1_compress(tau_g1).hex() == TAU_G1
    rng = random.Random(4844)
    hx = lambda b: b.hex()  # noqa: E731
    rand_fe = lambda: rng.randrange(ko.R)  # noqa: E731

    blobs = {}   # name -> (recipe, commitment, proof)
    for k in range(2):
        rec = {"random": f"kzg-golden-{k}"}
        blob = build_blob(rec)
        c = ko.blob_to_kzg_commitment(blob, g1_lagrange)
        blobs[f"full_{k}"] = (rec, c, ko.compute_blob_kzg_proof(blob, c, g1_lagrange))
    for k in range(4):
        a, b = rand_fe(), rand_fe()
        rec = {"deg1": [hex(a), hex(b)]}
        _, c, p = ko.degree1_case(a, b, tau_g1)
        blobs[f"deg1_{k}"] = (rec, c, p)
    rec0, c0, p0 = blobs["deg1_0"]
    rec1, c1, p1 = blobs["deg1_1"]
    flipped = bytearray(build_blob(rec0)[32 * 5:32 * 6])
    flipped[31] ^= 1
    if int.from_bytes(flipped, "big") >= ko.R:
        flipped[31] ^= 3
    blobs["flipped_element"] = (dict(rec0, edits={"5": hx(bytes(flipped))}), c0, p0)
    blobs["element_eq_r"] = (dict(rec0, edits={"7": hx(ko.R.to_bytes(32, "big"))}), c0, p0)
    blobs["element_r_minus_1"] = (dict(rec1, edits={"4095": hx((ko.R - 1).to_bytes(32, "big"))}), c1, p1)
    blobs["element_all_ones"] = (dict(rec1, edits={"9": "ff" * 32}), c1, p1)
    blobs["swapped_proofs"] = (blobs["full_0"][0], blobs["full_0"][1], blobs["full_1"][2])
    blobs["zero_blob_infinity"] = ({"zero": True}, ko.G1_INFINITY, ko.G1_INFINITY)
    blobs["zero_blob_wrong_proof"] = ({"zero": True}, ko.G1_INFINITY, p0)
    neg_c0 = bytearray(c0)
    neg_c0[0] ^= 0x20
    blobs["wrong_sign_commitment"] = (rec0, bytes(neg_c0), p0)
    x_ge_p = bytearray(bo.P.to_bytes(48, "big"))
    x_ge_p[0] |= 0x80
    blobs["commitment_x_ge_p"] = (rec0, bytes(x_ge_p), p0)
    blobs["proof_not_in_g1"] = (rec0, c0, off_subgroup_point())
    blobs["commitment_not_in_g1"] = (rec0, off_subgroup_point(), p0)
    uncompressed = bytearray(c0)
    uncompressed[0] &= 0x7F
    blobs["commitment_compression_bit_clear"] = (rec0, bytes(uncompressed), p0)
    blobs["proof_infinity_with_payload"] = (rec0, c0, bytes([0xC0]) + bytes(46) + b"\x01")

    blob_cases = []
    for name, (rec, c, p) in blobs.items():
        code = ko.verify_blob_kzg_proof(build_blob(rec), c, p, tau_g2)
        blob_cases.append({"name": name, "blob": rec, "commitment": hx(c), "proof": hx(p), "code": code})
    by_name = {c["name"]: c for c in blob_cases}
    assert by_name["full_0"]["code"] == by_name["deg1_0"]["code"] == by_name["zero_blob_infinity"]["code"] == 0

    # verify_kzg_proof: p(X) = a + bX at chosen z (proof [b]G1, y = a + bz), and the full-degree blobs at their challenges
    point_cases = []
    a, b = rand_fe(), rand_fe()
    _, c, p = ko.degree1_case(a, b, tau_g1)
    z = rand_fe()
    y = (a + b * z) % ko.R
    w3 = ko.ROOTS_BRP[3]
    pts = {"deg1_random_z": (c, z, y, p), "deg1_wrong_y": (c, z, y + 1, p), "deg1_z_in_domain": (c, w3, (a + b * w3) % ko.R, p),
           "z_eq_r": (c, ko.R, y, p), "y_eq_r": (c, z, ko.R, p), "y_r_minus_1": (c, z, ko.R - 1, p),
           "infinity_zero_poly": (ko.G1_INFINITY, z, 0, ko.G1_INFINITY), "infinity_nonzero_y": (ko.G1_INFINITY, z, 1, ko.G1_INFINITY),
           "proof_not_in_g1": (c, z, y, off_subgroup_point())}
    for k in range(2):
        rec, cf, pf = blobs[f"full_{k}"]
        blob = build_blob(rec)
        zf = ko.compute_challenge(blob, cf)
        pts[f"full_{k}_at_challenge"] = (cf, zf, ko.evaluate_polynomial_in_evaluation_form(ko.blob_to_polynomial(blob), zf), pf)
    for name, (c, z, y, p) in pts.items():
        zb, yb = z.to_bytes(32, "big"), y.to_bytes(32, "big")
        point_cases.append({"name": name, "commitment": hx(c), "z": hx(zb), "y": hx(yb), "proof": hx(p),
                            "code": ko.verify_kzg_proof(c, zb, yb, p, tau_g2)})

    # verify_blob_kzg_proof_batch over lists of blob cases
    batch_cases = []
    for name, members in (("all_valid", ["full_0", "full_1", "deg1_0", "deg1_1", "deg1_2", "deg1_3", "zero_blob_infinity"]),
                          ("one_invalid", ["full_0", "deg1_0", "flipped_element", "deg1_2"]),
                          ("swapped", ["full_0", "swapped_proofs"]),
                          ("bad_element", ["deg1_0", "element_eq_r", "deg1_1"]),
                          ("bad_point", ["deg1_2", "proof_not_in_g1"]),
                          ("single_valid", ["full_1"]), ("single_invalid", ["flipped_element"]), ("empty", [])):
        cs = [by_name[m] for m in members]
        code = ko.verify_blob_kzg_proof_batch([build_blob(c["blob"]) for c in cs], [bytes.fromhex(c["commitment"]) for c in cs],
                                              [bytes.fromhex(c["proof"]) for c in cs], tau_g2)
        batch_cases.append({"name": name, "members": members, "code": code})

    doc = {"tau_g1": TAU_G1, "blob_cases": blob_cases, "point_cases": point_cases, "batch_cases": batch_cases}
    parts = [f'"tau_g1": {json.dumps(TAU_G1)}'] + [f"{json.dumps(k)}: [\n" + ",\n".join(json.dumps(c) for c in doc[k]) + "\n]"
                                                  for k in ("blob_cases", "point_cases", "batch_cases")]
    out.write_text("{" + ",\n".join(parts) + "}\n")   # one case per line
    return doc


if __name__ == "__main__":
    main(Path(sys.argv[1]) if len(sys.argv) > 1 else OUT)
