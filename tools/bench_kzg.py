#!/usr/bin/env python
"""KZG blob-proof verification on one B200: one JSON line per batch size n of b200_verify_blob_kzg_proofs (one code per blob;
verify_blob_kzg_proof_batch is the same call reduced to one code).

`device_ms`: CUDA events on the library stream from the first kernel to the last (inputs already copied); `e2e_ms`: host
clock around the public call with blobs, commitments and proofs in pinned host buffers (H2D + kernels + D2H inside).
Medians over --steps timed calls after --warmup.  `stages_ms` is the B200_KZG_TRACE split of the last timed call.

Workload: degree-1 blobs on the mainnet trusted setup (valid by construction, oracle/kzg_oracle.py), a pool of 16 distinct
triples tiled to n.  Verification does the same work for every valid blob whatever its polynomial (4 096 elements
decoded and folded, 2 050 SHA-256 compressions, two 255-bit scalar multiplications, two Miller loops), so degree-1
fixtures are a fair workload.
Usage: python tools/bench_kzg.py [--sizes 1,6,64,512,4096] [--steps 5] [--warmup 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

FR_PRODUCTS_PER_BLOB = 4096 * 5 + 255 * 3 + 1   # per element: to Montgomery + four in the fraction fold; CTA tree; 1/4096
SHA256_COMPRESSIONS_PER_BLOB = 2050             # (32 + 131 072 + 48 + 9) bytes -> 2 050 blocks


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, _, limit = r.stdout.strip().partition(",")
    return name.strip(), limit.strip()


def traced(fn):
    """Runs fn() with fd 2 redirected to a file and returns the library's trace line."""
    with tempfile.TemporaryFile(mode="w+") as f:
        sys.stderr.flush()
        saved = os.dup(2)
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
        f.seek(0)
        lines = [ln for ln in f.read().splitlines() if ln.startswith("[b200 kzg]")]
    return lines[-1] if lines else ""


def parse_trace(line: str) -> dict:
    return {k: float(v) for k, v in re.findall(r"\| (\w+) ([0-9.]+)", line)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,6,64,512,4096")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    os.environ["B200_KZG_TRACE"] = "1"   # read once when the KZG path is first used; the timed calls below print nothing
    import torch

    from ethereum_consensus_b200 import _lib, kzg
    from oracle import bls_oracle as bo
    from oracle import kzg_oracle as ko

    lib = _lib.init(0)
    from tests.golden import make_kzg_golden as mk
    settings = kzg.kzg_settings_from_json(mk.setup_json())
    tau_g1 = bo.g1_uncompress(bytes.fromhex(mk.TAU_G1))[1]
    pool = [ko.degree1_case(1000 + 7 * i, 2000 + 13 * i, tau_g1) for i in range(16)]
    name, power = card()
    sizes = [int(s) for s in a.sizes.split(",")]
    nmax = max(sizes)
    pin = lambda data, n: torch.frombuffer(bytearray(b"".join(data[i % len(data)] for i in range(n))),  # noqa: E731
                                                  dtype=torch.uint8).pin_memory()
    blobs, comms, proofs = (pin([p[k] for p in pool], nmax) for k in range(3))
    out_lines = []
    for n in sizes:
        codes = np.zeros(n, np.int32)
        call = lambda: lib.b200_verify_blob_kzg_proofs(settings.handle, blobs.data_ptr(), comms.data_ptr(),  # noqa: E731
                                                       proofs.data_ptr(), n, codes.ctypes.data)
        for _ in range(a.warmup):
            traced(call)
        dev, e2e, line = [], [], ""
        for _ in range(a.steps):
            t = {}

            def timed():
                t0 = time.perf_counter()
                t["rc"] = call()
                t["ms"] = (time.perf_counter() - t0) * 1e3
            line = traced(timed)
            assert t["rc"] == 0 and not codes.any(), (n, t["rc"], np.unique(codes))
            dev.append(float(lib.b200_last_kernel_ms()))
            e2e.append(t["ms"])
        rec = {"n": n, "device_ms": float(np.median(dev)), "e2e_ms": float(np.median(e2e)),
               "blobs_per_s_device": n / (np.median(dev) / 1e3), "blobs_per_s_e2e": n / (np.median(e2e) / 1e3),
               "stages_ms": parse_trace(line), "steps": a.steps, "warmup": a.warmup,
               "work_per_blob": {"fr_products": FR_PRODUCTS_PER_BLOB, "sha256_compressions": SHA256_COMPRESSIONS_PER_BLOB,
                                 "h2d_bytes": kzg.BYTES_PER_BLOB + 96},
               "workload": "degree-1 mainnet-setup blobs (16 distinct, tiled); verification work does not depend on the polynomial",
               "card": name, "power_limit": power}
        print(json.dumps(rec), flush=True)
        out_lines.append(json.dumps(rec))
    if a.out:
        Path(a.out).write_text("\n".join(out_lines) + "\n")


if __name__ == "__main__":
    main()
