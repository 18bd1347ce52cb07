"""One rank of tests/test_config_scale_gpu.py::test_two_rank_sharded_calls_over_nccl (also runnable by hand on a
machine with two GPUs).  No torch: the library's communicator is created from a 128-byte id that rank 0 writes to a file —
the same bootstrap a Rust host would do over whatever channel it has."""
import ctypes as C
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from ethereum_consensus_b200 import _lib, crypto, parallel, ssz, state as S  # noqa: E402

rank, world = int(os.environ["B200_TEST_RANK"]), int(os.environ["B200_TEST_WORLD"])
box = Path(os.environ["B200_TEST_DIR"])
lib = _lib.init(int(os.environ.get("B200_TEST_DEVICE", "0")))
ident = (C.c_uint8 * 128)()
id_file = box / "nccl_id.bin"
if rank == 0:
    _lib.check(lib.b200_comm_unique_id(ident), "comm_unique_id")
    tmp = box / "nccl_id.tmp"
    tmp.write_bytes(bytes(ident))
    tmp.rename(id_file)
else:
    t0 = time.time()
    while not id_file.exists():
        if time.time() - t0 > 120:
            raise SystemExit("timed out waiting for the NCCL id")
        time.sleep(0.05)
    C.memmove(ident, id_file.read_bytes(), 128)
_lib.check(lib.b200_comm_init(ident, rank, world), "comm_init")
assert parallel.comm_info()[:2] == (rank, world)

# ---- SSZ: ragged sizes so that slices are uneven / empty on the last rank
for n in (1, 5, 70_001, 1 << 17):
    st = S.synth_state(n, "mainnet", n_historical_summaries=3, n_historical_roots=2)
    ser = S.serialize(st)
    want = ssz.hash_tree_root_beacon_state(ser, "mainnet")
    got = parallel.sharded_state_root(ser, "mainnet")
    assert got == want, (n, got.hex(), want.hex())
    if n == 70_001:   # resident across the ranks: root is kernels + one all-gather
        dev = ssz.DeviceBeaconState(ser, "mainnet", sharded=True)
        assert dev.hash_tree_root() == want and dev.hash_tree_root() == want
        dev.close()
st = S.synth_state(300, "minimal", n_historical_summaries=3, n_historical_roots=2)
ser = S.serialize(st)
assert parallel.sharded_state_root(ser, "minimal") == ssz.hash_tree_root_beacon_state(ser, "minimal")

# ---- BLS: the golden batch (every reject class) through the sharded call: all verdicts on every rank
cases = [c for c in json.loads((ROOT / "tests" / "golden" / "bls_cases.json").read_text())["fast_aggregate_verify"] if len(c["msg"]) == 64]
for reps in (1, 3):
    cs = cases * reps
    pks = np.frombuffer(b"".join(bytes.fromhex(p) for c in cs for p in c["pks"]), dtype=np.uint8)
    off = np.cumsum([0] + [len(c["pks"]) for c in cs]).astype(np.uint32)
    msgs = np.frombuffer(b"".join(bytes.fromhex(c["msg"]) for c in cs), dtype=np.uint8)
    sigs = np.frombuffer(b"".join(bytes.fromhex(c["sig"]) for c in cs), dtype=np.uint8)
    got = parallel.sharded_verify_batch(pks, off, msgs, sigs)
    assert got.tolist() == [c["code"] for c in cs], got.tolist()
one = parallel.sharded_verify_batch(pks[: 48 * int(off[1])], off[:2], msgs[:32], sigs[:96])   # fewer tuples than ranks
assert one.tolist() == [cases[0]["code"]]
# ---- RLC whole-batch check over both ranks: Gt / G2 partials travel in one ncclAllGather
import hashlib  # noqa: E402
good = [c for c in cases if c["code"] == 0] * 3
gp = np.frombuffer(b"".join(bytes.fromhex(p) for c in good for p in c["pks"]), dtype=np.uint8)
go = np.cumsum([0] + [len(c["pks"]) for c in good]).astype(np.uint32)
gm = np.frombuffer(b"".join(bytes.fromhex(c["msg"]) for c in good), dtype=np.uint8)
gs = np.frombuffer(b"".join(bytes.fromhex(c["sig"]) for c in good), dtype=np.uint8).copy()
seed = hashlib.sha256(b"two ranks").digest()
assert crypto.fast_aggregate_verify_batch_all(gp, go, gm, gs, seed=seed, sharded=True) is True
gs_bad = gs.copy(); gs_bad[-96:] = gs[:96]      # the LAST tuple (rank 1's block) carries the first tuple's signature
assert crypto.fast_aggregate_verify_batch_all(gp, go, gm, gs_bad, seed=seed, sharded=True) is False
gs_bad = gs.copy(); gs_bad[:96] = gs[-96:]      # ... and a failure in rank 0's block is seen by rank 1 as well
assert crypto.fast_aggregate_verify_batch_all(gp, go, gm, gs_bad, seed=seed, sharded=True) is False
mine = np.array([rank * 10 + 1, rank * 10 + 2], dtype=np.int32)
assert parallel.comm_all_gather_codes(mine).tolist() == [r * 10 + k for r in range(world) for k in (1, 2)]
assert lib.b200_collective_count() > 0
parallel.comm_destroy()
print("SHARDED_OK rank", rank, "collectives", lib.b200_collective_count(), flush=True)
