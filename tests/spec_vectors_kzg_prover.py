"""The prover handlers of the conformance-vector runner (the reference's spec-tests/runners/kzg.rs):
`tests/<config>/deneb/kzg/<handler>/<suite>/<case>/data.yaml`.  A case passes when the call's output equals `output`
byte for byte, or, with `output: null`, when the input does not deserialize or the call fails.  `compute_kzg_proof`'s
output is the pair [proof, y].  The verification handlers are in spec_vectors_kzg.py.  Test infrastructure only."""
from __future__ import annotations

from pathlib import Path
from typing import Tuple

from tests.spec_vectors import unhex
from tests.spec_vectors_kzg import BYTES_PER_BLOB, write_case

KZG_PROVER_HANDLERS = ("blob_to_kzg_commitment", "compute_kzg_proof", "compute_blob_kzg_proof")


def run_kzg_prover_case(handler: str, case_dir: Path, impl) -> Tuple[bool, str]:
    import yaml
    d = yaml.safe_load((case_dir / "data.yaml").read_text())
    inp, want = d["input"], d["output"]
    if handler == "blob_to_kzg_commitment":
        args = [unhex(inp.get("blob"), BYTES_PER_BLOB)]
    elif handler == "compute_kzg_proof":
        args = [unhex(inp.get("blob"), BYTES_PER_BLOB), unhex(inp.get("z"), 32)]
    elif handler == "compute_blob_kzg_proof":
        args = [unhex(inp.get("blob"), BYTES_PER_BLOB), unhex(inp.get("commitment"), 48)]
    else:
        raise ValueError(handler)
    if any(a is None for a in args):
        return want is None, "malformed input"
    try:
        got = getattr(impl, handler)(*args)
    except impl.Error:
        return want is None, "call failed"
    if want is None:
        return False, "expected a failure"
    if handler == "compute_kzg_proof":
        return [bytes(x) for x in got] == [unhex(want[0], 48), unhex(want[1], 32)], ""
    return bytes(got) == unhex(want, 48), ""


class OracleKzgProverImpl:
    """tests/kzg_prover_oracle.py behind the prover call surface (g1_lagrange bound at construction)."""

    class Error(Exception):
        pass

    def __init__(self, setup: dict):
        from oracle import kzg_oracle as ko
        from tests import kzg_prover_oracle as kp
        self.ko, self.kp = ko, kp
        self.g1 = ko.load_setup(setup)[0]

    def _ok(self, code, *out):
        if code != 0:
            raise self.Error(code)
        return out[0] if len(out) == 1 else out

    def blob_to_kzg_commitment(self, b): return self._ok(*self.kp.blob_to_kzg_commitment_code(b, self.g1))
    def compute_kzg_proof(self, b, z): return self._ok(*self.kp.compute_kzg_proof_code(b, z, self.g1))
    def compute_blob_kzg_proof(self, b, c): return self._ok(*self.kp.compute_blob_kzg_proof_code(b, c, self.g1))


class DeviceKzgProverImpl:
    """ethereum_consensus_b200.kzg's prover with one loaded settings handle."""

    def __init__(self, settings):
        from ethereum_consensus_b200 import kzg
        self.kzg, self.s, self.Error = kzg, settings, kzg.Error

    def blob_to_kzg_commitment(self, b): return self.kzg.blob_to_kzg_commitment(b, self.s)

    def compute_kzg_proof(self, b, z):
        r = self.kzg.compute_kzg_proof(b, z, self.s)
        return r.proof, r.evaluation

    def compute_blob_kzg_proof(self, b, c): return self.kzg.compute_blob_kzg_proof(b, c, self.s)


def synthetic_prover_tree(base: Path, golden: dict, build_blob, names=None) -> Path:
    """Prover golden cases (kzg_prover_cases.json) in the consensus-spec-tests layout, plus literals that do not
    deserialize.  `names`: only the cases with these names (the oracle runs an MSM per valid case)."""
    hx = lambda b: "0x" + (b if isinstance(b, str) else b.hex())  # noqa: E731
    keep = lambda c: names is None or c["name"] in names  # noqa: E731
    for c in filter(keep, golden["commit_cases"]):
        write_case(base, "blob_to_kzg_commitment", c["name"], {"blob": hx(build_blob(c["blob"]))},
                   None if c["code"] else hx(c["commitment"]))
    for c in filter(keep, golden["point_cases"]):
        write_case(base, "compute_kzg_proof", c["name"], {"blob": hx(build_blob(c["blob"])), "z": hx(c["z"])},
                   None if c["code"] else [hx(c["proof"]), hx(c["y"])])
    for c in filter(keep, golden["blob_cases"]):
        write_case(base, "compute_blob_kzg_proof", c["name"], {"blob": hx(build_blob(c["blob"])), "commitment": hx(c["commitment"])},
                   None if c["code"] else hx(c["proof"]))
    write_case(base, "blob_to_kzg_commitment", "case_short_blob", {"blob": "0x00"}, None)
    write_case(base, "compute_kzg_proof", "case_short_z", {"blob": hx(bytes(BYTES_PER_BLOB)), "z": "0x1234"}, None)
    write_case(base, "compute_blob_kzg_proof", "case_short_commitment", {"blob": hx(bytes(BYTES_PER_BLOB)), "commitment": "0xc0"}, None)
    return base
