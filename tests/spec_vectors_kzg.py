"""KZG half of the conformance-vector runner: the verification handlers of the reference's spec-tests/runners/kzg.rs
(`tests/<config>/deneb/kzg/<handler>/<suite>/<case>/data.yaml` with `input` and `output`).  As in that runner, an input
literal that does not deserialize (wrong length, not hex) means the case expects `output: null`; otherwise the call must
succeed exactly when `output` is true.  The prover handlers (blob_to_kzg_commitment, compute_*) are out of scope here.
Test infrastructure only."""
from __future__ import annotations

from pathlib import Path
from typing import Tuple

import yaml

from tests.spec_vectors import unhex

KZG_HANDLERS = ("verify_kzg_proof", "verify_blob_kzg_proof", "verify_blob_kzg_proof_batch")
BYTES_PER_BLOB = 131072


def run_kzg_case(handler: str, case_dir: Path, impl) -> Tuple[bool, str]:
    d = yaml.safe_load((case_dir / "data.yaml").read_text())
    inp, want = d["input"], d["output"]

    def ok(fn, *a):
        try:
            fn(*a)
            return True
        except impl.Error:
            return False

    if handler == "verify_kzg_proof":
        args = [unhex(inp.get("commitment"), 48), unhex(inp.get("z"), 32), unhex(inp.get("y"), 32), unhex(inp.get("proof"), 48)]
        if any(a is None for a in args):
            return want is None, "malformed input"
        return ok(impl.verify_kzg_proof, *args) == (want is True), ""
    if handler == "verify_blob_kzg_proof":
        args = [unhex(inp.get("blob"), BYTES_PER_BLOB), unhex(inp.get("commitment"), 48), unhex(inp.get("proof"), 48)]
        if any(a is None for a in args):
            return want is None, "malformed input"
        return ok(impl.verify_blob_kzg_proof, *args) == (want is True), ""
    if handler == "verify_blob_kzg_proof_batch":
        blobs = [unhex(b, BYTES_PER_BLOB) for b in inp.get("blobs") or []]
        cs = [unhex(c, 48) for c in inp.get("commitments") or []]
        ps = [unhex(p, 48) for p in inp.get("proofs") or []]
        if any(x is None for x in blobs + cs + ps):
            return want is None, "malformed input"
        return ok(impl.verify_blob_kzg_proof_batch, blobs, cs, ps) == (want is True), ""
    raise ValueError(handler)


class OracleKzgImpl:
    """oracle/kzg_oracle.py behind the call surface of ethereum_consensus_b200.kzg (settings bound at construction)."""

    class Error(Exception):
        pass

    def __init__(self, setup: dict):
        from oracle import bls_oracle as bo
        from oracle import kzg_oracle as ko
        self.ko = ko
        self.tau_g2 = bo.g2_uncompress(bytes.fromhex(setup["g2_monomial"][1][2:]))[1]

    def _chk(self, code):
        if code != 0:
            raise self.Error(code)

    def verify_kzg_proof(self, c, z, y, p): self._chk(self.ko.verify_kzg_proof(c, z, y, p, self.tau_g2))
    def verify_blob_kzg_proof(self, b, c, p): self._chk(self.ko.verify_blob_kzg_proof(b, c, p, self.tau_g2))
    def verify_blob_kzg_proof_batch(self, bs, cs, ps): self._chk(self.ko.verify_blob_kzg_proof_batch(bs, cs, ps, self.tau_g2))


class DeviceKzgImpl:
    """ethereum_consensus_b200.kzg with one loaded settings handle."""

    def __init__(self, settings):
        from ethereum_consensus_b200 import kzg
        self.kzg, self.s, self.Error = kzg, settings, kzg.Error

    def verify_kzg_proof(self, c, z, y, p): self.kzg.verify_kzg_proof(c, z, y, p, self.s)
    def verify_blob_kzg_proof(self, b, c, p): self.kzg.verify_blob_kzg_proof(b, c, p, self.s)
    def verify_blob_kzg_proof_batch(self, bs, cs, ps): self.kzg.verify_blob_kzg_proof_batch(bs, cs, ps, self.s)


def write_case(base: Path, handler: str, name: str, inp, out) -> None:
    d = base / "tests" / "general" / "deneb" / "kzg" / handler / "kzg-mainnet" / name
    d.mkdir(parents=True, exist_ok=True)
    (d / "data.yaml").write_text(yaml.safe_dump({"input": inp, "output": out}))


def synthetic_tree(base: Path, golden: dict, build_blob, max_blob_cases: int = 8) -> Path:
    """Golden cases re-expressed in the consensus-spec-tests layout, plus literals that do not deserialize."""
    hx = lambda b: "0x" + (b if isinstance(b, str) else b.hex())  # noqa: E731
    for c in golden["point_cases"]:
        write_case(base, "verify_kzg_proof", c["name"], {k: hx(c[k]) for k in ("commitment", "z", "y", "proof")},
                   None if c["code"] == 17 else c["code"] == 0)
    by_name = {c["name"]: c for c in golden["blob_cases"]}
    picked = [c for c in golden["blob_cases"] if not c["name"].startswith("full_")][:max_blob_cases]
    for c in picked:
        write_case(base, "verify_blob_kzg_proof", c["name"], {"blob": hx(build_blob(c["blob"])), "commitment": hx(c["commitment"]),
                                                              "proof": hx(c["proof"])}, None if c["code"] == 17 else c["code"] == 0)
    for c in golden["batch_cases"]:
        ms = [by_name[m] for m in c["members"]]
        if any(m["name"].startswith("full_") for m in ms):
            continue
        write_case(base, "verify_blob_kzg_proof_batch", c["name"],
                   {"blobs": [hx(build_blob(m["blob"])) for m in ms], "commitments": [hx(m["commitment"]) for m in ms],
                    "proofs": [hx(m["proof"]) for m in ms]}, None if c["code"] == 17 else c["code"] == 0)
    ok = by_name["deg1_0"]
    write_case(base, "verify_blob_kzg_proof", "case_short_blob", {"blob": "0x00", "commitment": hx(ok["commitment"]),
                                                                  "proof": hx(ok["proof"])}, None)
    pc = golden["point_cases"][0]
    write_case(base, "verify_kzg_proof", "case_short_z", {"commitment": hx(pc["commitment"]), "z": "0x1234", "y": hx(pc["y"]),
                                                          "proof": hx(pc["proof"])}, None)
    write_case(base, "verify_blob_kzg_proof_batch", "case_length_mismatch",
               {"blobs": [hx(build_blob(ok["blob"]))], "commitments": [], "proofs": [hx(ok["proof"])]}, None)
    return base
