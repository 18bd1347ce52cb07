#!/usr/bin/env python
"""deneb epoch processing on one B200, on the config-3 state (2**20 validators, mainnet preset): JSON lines.

Rows (`op`):
  * `stage`: one process_epoch stage alone (stage_mask = one bit), host clock around the call (the call ends in a
    stream synchronize, so this is launches + kernels + the host logic of that stage).
  * `epoch`: process_epoch with every stage at a plain epoch, then the first b200_state_root_incremental after it
    (the lists are whole-chain dirty, so it is a full re-hash) and, for comparison, b200_state_root.
  * `slots`: process_slots from the last slot of an epoch across the boundary (one state root, the epoch, the writes).
  * `eth1_boundary` / `sync_boundary`: process_epoch at the two period boundaries (the eth1_data_votes reset and its
    re-layout; historical_summaries + sync committee from real registry keys, tiled from 2**15 distinct ones as in
    tests/workloads.py).
  * `oracle`: the numpy oracle (oracle/epoch_oracle.py) on the host for the same plain epoch.
`bytes_min` is the HBM traffic the per-validator sweeps need (records read once per sweep, lists read and written), and
`hbm_share` its time at 7.7 TB/s over the measured epoch time.  Medians over --steps after --warmup; each timed call
runs on a freshly uploaded state.  The card name and power limit are read in the same run.
Usage: python tools/bench_epoch.py [--n 1048576] [--steps 5] [--warmup 1] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes
import hashlib
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True

HBM_BYTES_PER_S = 7.7e12


def card():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power = (r.stdout.strip().split(", ") + ["?"])[:2]
    return name, power


def sweep_bytes(n: int) -> int:
    """sums (records + two flag lists), rewards (records, balances r/w, flags, scores r/w), registry marking (records),
    slashings + effective balances (records, balances r/w), participation rotation (copy + clear)"""
    rec = 121 * n
    return (rec + 2 * n) + (rec + 16 * n + n + 16 * n) + rec + (rec + 16 * n) + 3 * n


def state_for(n: int, kind: str, keys=None):
    from tests.golden import make_epoch_golden as mk
    from oracle import epoch_oracle as eo
    C = eo.CONSTS["mainnet"]
    e = {"plain": mk.plain_epoch("mainnet", 269_500), "eth1": mk.boundary_epoch("mainnet", "eth1", 269_500),
         "sync": mk.boundary_epoch("mainnet", "sync", 269_500)}[kind]
    st = mk.base_state("mainnet", n, e, 0xB200)
    rng = np.random.default_rng(7)
    v = st.validators
    v["effective_balance"] = (rng.integers(15, 33, n) * 10**9).astype(np.uint64)
    v["slashed"] = rng.integers(0, 512, n) == 0
    v["withdrawable_epoch"] = np.where(v["slashed"], e + C["EPOCHS_PER_SLASHINGS_VECTOR"] // 2, mk.FF)
    v["exit_epoch"] = np.where(v["slashed"], e + 5, mk.FF)
    st.slashings[::7] = 10**9
    st.balances = (v["effective_balance"] + rng.integers(0, 2 * 10**9, n)).astype("<u8")
    if keys is not None:
        v["public_key"] = np.resize(keys, (n, 48)).view("V48").reshape(n)
    return st


def real_keys(n_distinct: int = 1 << 15):
    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle")], check=True)
    orc = ctypes.CDLL(str(ROOT / "oracle" / "liboracle_bls.so"))
    orc.orc_pk_sequence.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p]
    r = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
    sk0 = int.from_bytes(hashlib.sha256(b"b200/sk0").digest(), "big") % r
    delta = int.from_bytes(hashlib.sha256(b"b200/delta").digest(), "big") % r
    keys = np.empty((n_distinct, 48), np.uint8)
    orc.orc_pk_sequence(sk0.to_bytes(32, "big"), delta.to_bytes(32, "big"), n_distinct, keys.ctypes.data)
    return keys


def timed(ssz_bytes, fn, steps, warmup):
    from ethereum_consensus_b200 import ssz
    out = []
    for k in range(warmup + steps):
        dev = ssz.DeviceBeaconState(ssz_bytes, "mainnet")
        t0 = time.perf_counter()
        extra = fn(dev)
        dt = (time.perf_counter() - t0) * 1e3
        if k >= warmup:
            out.append((dt, extra))
        dev.close()
    ms = sorted(x[0] for x in out)[len(out) // 2]
    return ms, [x[1] for x in out]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from ethereum_consensus_b200 import _lib, epoch
    from ethereum_consensus_b200 import state as S
    from oracle import epoch_oracle as eo
    _lib.init(0)
    name, power = card()
    rows = []

    def emit(row):
        row.update(card=name, power_limit=power, n=a.n, preset="mainnet", steps=a.steps)
        rows.append(row)
        print(json.dumps(row), flush=True)

    plain = S.serialize(state_for(a.n, "plain"))
    for bit, stage in enumerate(eo.STAGES):
        ms, _ = timed(plain, lambda d, b=bit: epoch.process_epoch(d, 1 << b), a.steps, a.warmup)
        emit({"op": "stage", "stage": stage, "call_ms": round(ms, 3)})

    def epoch_then_roots(d):
        epoch.process_epoch(d)
        t0 = time.perf_counter()
        d.hash_tree_root_incremental()
        t1 = time.perf_counter()
        d.hash_tree_root()
        t2 = time.perf_counter()
        return (t1 - t0) * 1e3, (t2 - t1) * 1e3
    ms, extra = timed(plain, epoch_then_roots, a.steps, a.warmup)
    inc = sorted(x[0] for x in extra)[len(extra) // 2]
    full = sorted(x[1] for x in extra)[len(extra) // 2]
    b = sweep_bytes(a.n)
    emit({"op": "epoch", "call_ms": round(ms, 3), "first_incremental_root_ms": round(inc, 3), "full_root_ms": round(full, 3),
          "bytes_min": b, "hbm_share": round(b / HBM_BYTES_PER_S * 1e3 / ms, 4)})

    slot = int.from_bytes(S.serialize(state_for(8, "plain"))[40:48].tobytes(), "little")
    ms, _ = timed(plain, lambda d: epoch.process_slots(d, slot + 1), a.steps, a.warmup)
    emit({"op": "slots", "from_slot": slot, "to_slot": slot + 1, "call_ms": round(ms, 3)})

    ms, _ = timed(S.serialize(state_for(a.n, "eth1")), lambda d: epoch.process_epoch(d), a.steps, a.warmup)
    emit({"op": "eth1_boundary", "call_ms": round(ms, 3)})
    ms, _ = timed(S.serialize(state_for(a.n, "sync", real_keys())), lambda d: epoch.process_epoch(d), a.steps, a.warmup)
    emit({"op": "sync_boundary", "call_ms": round(ms, 3)})

    st = state_for(a.n, "plain")
    t0 = time.perf_counter()
    rc = eo.process_epoch_numpy(st)
    emit({"op": "oracle", "host_ms": round((time.perf_counter() - t0) * 1e3, 1), "code": rc})
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text("".join(json.dumps(r) + "\n" for r in rows))


if __name__ == "__main__":
    main()
