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

`--op commit` / `--op prove` time the prover instead (b200_blob_to_kzg_commitments / b200_compute_blob_kzg_proofs) on seeded
uniform blobs (every element below 2^254; the work of the MSM does not depend on the values beyond the rare zero digit),
with the commitments for `prove` made once by the device before timing.  Those rows add the MSM's algorithmic work per blob
(Fp products from the window parameters, 288 32-bit multiply-adds each) and its rate over the `msm` stage time as a share
of the 9.31 T MAD/s integer issue rate of DESIGN.md §4.
Usage: python tools/bench_kzg.py [--op verify|commit|prove] [--sizes 1,6,64,512,4096] [--steps 5] [--warmup 2] [--out FILE]
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
# the MSM (csrc/msm.cuh): c = 5, 52 windows, 2 window groups per base, 128-thread CTAs -> 64 partial sums per blob
MSM_C, MSM_WINDOWS, MSM_GROUPS, MSM_CTA = 5, 52, 2, 128
MAD_PER_FP_PRODUCT = 288                        # 12 x 12 limb products + 12 x 12 for the reduction
INT_MAD_PER_S = 9.31e12                          # DESIGN.md §4: the B200's 32-bit IMAD issue rate


def msm_work_per_blob() -> dict:
    """Fp products of one blob's MSM for uniform scalars: a nonzero digit costs one mixed addition (11 products); the
    top window only ever holds the recoding carry (probability ~1/2^c); the CTA trees and the final tree add 16 each."""
    p_nonzero = 1 - 1 / (1 << MSM_C)
    mixed = 4096 * ((MSM_WINDOWS - 1) * p_nonzero + 1 / (1 << MSM_C))
    ctas = 4096 * MSM_GROUPS // MSM_CTA
    tree = ctas * (MSM_CTA - 1) + (ctas - 1)
    products = mixed * 11 + tree * 16
    return {"mixed_additions": round(mixed), "jacobian_additions": tree, "fp_products": round(products),
            "mads": round(products * MAD_PER_FP_PRODUCT)}


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
    ap.add_argument("--op", default="verify", choices=["verify", "commit", "prove"])
    a = ap.parse_args()
    if a.op != "verify":
        return prover(a)
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


def prover(a):
    os.environ["B200_KZG_TRACE"] = "1"
    import torch

    from ethereum_consensus_b200 import _lib, kzg
    from tests.golden import make_kzg_golden as mk

    lib = _lib.init(0)
    settings = kzg.kzg_settings_from_json(mk.setup_json())
    name, power = card()
    sizes = [int(s) for s in a.sizes.split(",")]
    nmax = max(sizes)
    rng = np.random.default_rng(4844)
    raw = rng.integers(0, 256, size=(nmax * 4096, 32), dtype=np.uint8)
    raw[:, 0] &= 0x3F                                  # every element < 2^254 < r
    blobs = torch.from_numpy(raw.reshape(-1)).pin_memory()
    comms = torch.zeros(nmax * 48, dtype=torch.uint8).pin_memory()
    outs = np.zeros((nmax, 48), np.uint8)
    if a.op == "prove":
        c, codes = kzg.blob_to_kzg_commitments(blobs, settings)
        assert not codes.any()
        comms.copy_(torch.from_numpy(c.reshape(-1)))
    work = msm_work_per_blob()
    out_lines = []
    for n in sizes:
        codes = np.zeros(n, np.int32)
        if a.op == "commit":
            call = lambda: lib.b200_blob_to_kzg_commitments(settings.handle, blobs.data_ptr(), n, outs.ctypes.data,  # noqa: E731
                                                            codes.ctypes.data)
        else:
            call = lambda: lib.b200_compute_blob_kzg_proofs(settings.handle, blobs.data_ptr(), comms.data_ptr(), n,  # noqa: E731
                                                            outs.ctypes.data, codes.ctypes.data)
        for _ in range(a.warmup):
            traced(call)
        dev, e2e, msm, line = [], [], [], ""
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
            msm.append(parse_trace(line).get("msm", float("nan")))
        msm_ms = float(np.median(msm))
        mad_rate = work["mads"] * n / (msm_ms / 1e3)
        rec = {"op": a.op, "n": n, "device_ms": float(np.median(dev)), "e2e_ms": float(np.median(e2e)),
               "blobs_per_s_device": n / (np.median(dev) / 1e3), "blobs_per_s_e2e": n / (np.median(e2e) / 1e3),
               "stages_ms": parse_trace(line), "steps": a.steps, "warmup": a.warmup,
               "msm_work_per_blob": work, "msm_ms": msm_ms, "msm_mad_per_s": mad_rate,
               "msm_share_of_int_issue_rate": mad_rate / INT_MAD_PER_S,
               "workload": "seeded uniform blobs, every element < 2^254" + ("; commitments made by the device before timing"
                                                                          if a.op == "prove" else ""),
               "card": name, "power_limit": power}
        print(json.dumps(rec), flush=True)
        out_lines.append(json.dumps(rec))
    if a.out:
        Path(a.out).write_text("\n".join(out_lines) + "\n")


if __name__ == "__main__":
    main()
