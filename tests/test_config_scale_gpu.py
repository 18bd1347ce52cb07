"""Parity at BASELINE.json's FULL config sizes (round-1 review: "config-scale parity lived in bench.py asserts"):

* configs[1]: T = 4096 tuples x K = 512 keys, strict — the exact workload bench.py times (tests/workloads.py) — against
  the C oracle on >= 1024 tuples + EVERY adversarial tuple, and registry mode + the sharded entry point on the same batch;
* configs[2]: hash_tree_root(BeaconState) at 2**20 validators against the hashlib golden root and the C oracle;
* configs[3]: the deneb process_block signature set at spec shape (K = 512 attestations, 16 slashings / exits /
  changes / deposits, K = 2048 attester slashings, 2**20-key registry), strict AND registry (`…_batch_indexed`) mode,
  bit-exact against the C oracle, with the reference's first-failure / deposit-tolerance replay;
* configs[4]: the library's sharded entry points at world = 1 here, and on 2 GPUs when the box has them.
"""
import ctypes
import hashlib
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

from ethereum_consensus_b200 import block, crypto, parallel, signing, ssz, state as S
from tests import workloads

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent


def _threads():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return os.cpu_count() or 1


@pytest.fixture(scope="module")
def comm1(engine):
    parallel.comm_init(0, 1)
    return parallel.comm_info()


@pytest.fixture(scope="module")
def config1(oracle_bls_c):
    return workloads.make_bls_workload(oracle_bls_c, 4096, 512, 0, threads=_threads())


def test_configs1_T4096_K512_strict_vs_c_oracle(engine, oracle_bls_c, config1):
    w, orc = config1, oracle_bls_c
    T, K = w["T"], w["K"]
    got = crypto.fast_aggregate_verify_batch(w["pks"], w["off"], w["msgs"], w["sigs"])
    assert got.tolist() == w["expect"].tolist()
    assert len(set(w["kind"].tolist())) == 6, "the workload must contain every adversarial kind"
    # C oracle: the first 1024 tuples as one multi-threaded batch ...
    n = 1024
    want = np.empty(n, dtype=np.int32)
    orc.orc_fast_aggregate_verify_batch(w["pks"].ctypes.data, w["off"].ctypes.data, w["msgs"].ctypes.data, w["sigs"].ctypes.data, n,
                                        want.ctypes.data, _threads())
    assert got[:n].tolist() == want.tolist()
    # ... and every adversarial tuple of the whole batch
    bad = np.nonzero(w["kind"] != 0)[0]
    sub_off = np.concatenate([[0], np.cumsum(np.full(len(bad), K))]).astype(np.uint32)
    pk = w["pks"].reshape(T, K * 48)[bad].reshape(-1).copy()
    ms = w["msgs"].reshape(T, 32)[bad].reshape(-1).copy()
    sg = w["sigs"].reshape(T, 96)[bad].reshape(-1).copy()
    want_bad = np.empty(len(bad), dtype=np.int32)
    orc.orc_fast_aggregate_verify_batch(pk.ctypes.data, sub_off.ctypes.data, ms.ctypes.data, sg.ctypes.data, len(bad), want_bad.ctypes.data,
                                        _threads())
    assert got[bad].tolist() == want_bad.tolist()


def test_configs1_registry_mode_same_verdicts(engine, config1):
    w = config1
    reg = crypto.Registry(w["registry"])
    assert (reg.key_codes() == 0).all()
    got = reg.verify_batch(w["idx"], w["off"], w["msgs"], w["sigs"])
    same = (w["kind"] != 4) & (w["kind"] != 5)   # those two kinds edit key BYTES, which index mode never sees
    assert got[same].tolist() == w["expect"][same].tolist()


def test_configs4_sharded_entry_point_world1(engine, comm1, config1):
    assert comm1[:2] == (0, 1)
    w = config1
    n = 2048                                       # configs[4]: one epoch's 32 x 64 tuples
    got = parallel.sharded_verify_batch(w["pks"][: n * 512 * 48], w["off"][: n + 1], w["msgs"][: 32 * n], w["sigs"][: 96 * n])
    assert got.tolist() == w["expect"][:n].tolist()
    assert parallel.comm_all_gather_codes(got).tolist() == got.tolist()


def test_configs2_full_state_root(engine, comm1, oracle_ssz_c):
    st = S.synth_state(1 << 20, "mainnet")
    ser = S.serialize(st)
    golden = json.loads((ROOT / "tests" / "golden" / "ssz_roots.json").read_text())["mainnet:1048576:default"]
    root = ssz.hash_tree_root_beacon_state(ser, "mainnet")
    assert root.hex() == golden
    out = ctypes.create_string_buffer(32)
    assert oracle_ssz_c.orc_htr_beacon_state_deneb(ser.ctypes.data, len(ser), 0, _threads(), out) == 0
    assert out.raw == root
    assert parallel.sharded_state_root(ser, "mainnet") == root          # exchange plumbing at world = 1
    sdev = ssz.DeviceBeaconState(ser, "mainnet", sharded=True)          # ... and resident across the (one) rank
    assert sdev.hash_tree_root() == root
    sdev.close()
    dev = ssz.DeviceBeaconState(ser, "mainnet")
    assert dev.hash_tree_root() == root
    dev.close()


def test_configs3_block_signature_set_spec_shape(engine, oracle_bls_c):
    orc = oracle_bls_c
    registry, rows = workloads.make_deneb_block_plan(orc, threads=_threads())
    assert len(rows) == 215
    s = workloads.collect_block_signature_set(registry, rows)
    strict = s.verify()
    assert strict.tolist() == [r["expect"] for r in rows]

    # the C oracle on the identical tuples, bit for bit
    want = np.empty(len(rows), dtype=np.int32)
    flat = np.frombuffer(b"".join(p for e in s.entries for p in e.pubkeys), dtype=np.uint8)
    off = np.cumsum([0] + [len(e.pubkeys) for e in s.entries]).astype(np.uint32)
    msgs = np.frombuffer(b"".join(e.signing_root for e in s.entries), dtype=np.uint8)
    sg = np.frombuffer(b"".join(e.signature for e in s.entries), dtype=np.uint8)
    orc.orc_fast_aggregate_verify_batch(flat.ctypes.data, off.ctypes.data, msgs.ctypes.data, sg.ctypes.data, len(rows), want.ctypes.data, _threads())
    assert strict.tolist() == want.tolist()

    # registry mode (`…_batch_indexed` for the 183 index-named checks, strict for deposits / bls changes): same vector
    reg = crypto.Registry(registry.reshape(-1))
    assert s.verify(registry=reg).tolist() == strict.tolist()
    dep = [i for i, r in enumerate(rows) if r["site"] == "deposit"]
    assert s.first_failure(strict) is None and s.skipped_deposits(strict) == [dep[3], dep[7]]
    # an invalid attestation aborts the block there; a later failure is never reported
    att = [i for i, r in enumerate(rows) if r["site"] == "attestation"]
    s.entries[att[70]].signature = s.entries[att[71]].signature
    s.entries[-1].signature = s.entries[0].signature
    for codes in (s.verify(), s.verify(registry=reg)):
        assert s.first_failure(codes) == (att[70], "attestation", 5)


def test_get_domain_and_sync_aggregate_signing_root(engine):
    """phase0/helpers.rs:190-222 + altair/block_processing.rs:216-243 vs the hashlib oracle."""
    from oracle import ssz_oracle as so
    gvr = hashlib.sha256(b"gvr").digest()
    fork = signing.Fork(bytes.fromhex("03000000"), bytes.fromhex("04000000"), 100)
    for epoch, version in ((99, "03000000"), (100, "04000000"), (101, "04000000")):
        d = signing.get_domain(fork, gvr, signing.DomainType.BeaconAttester, epoch)
        assert d == so.compute_domain(bytes.fromhex("01000000"), bytes.fromhex(version), gvr)
    assert signing.get_domain(fork, gvr, signing.DomainType.Randao, current_epoch=100) == \
        so.compute_domain(bytes.fromhex("02000000"), bytes.fromhex("04000000"), gvr)
    # first slot after the fork boundary: the sync aggregate signs slot - 1, i.e. the PREVIOUS fork version's domain
    s = block.SignatureSet()
    prev_root = hashlib.sha256(b"block root").digest()
    keys = [bytes([0xC0]) + bytes(47)] * 4
    s.add_sync_aggregate(keys, [True, False, True, True], crypto.INFINITY_COMPRESSED_SIGNATURE, 100 * 32, prev_root, fork, gvr)
    d_prev = so.compute_domain(bytes.fromhex("07000000"), bytes.fromhex("03000000"), gvr)
    assert s.entries[0].signing_root == so.compute_signing_root(prev_root, d_prev)
    assert len(s.entries[0].pubkeys) == 3 and s.entries[0].eth_variant
    s2 = block.SignatureSet()
    s2.add_sync_aggregate(keys, [False] * 4, crypto.INFINITY_COMPRESSED_SIGNATURE, 0, prev_root, fork, gvr)   # slot 0 -> previous_slot 0
    assert s2.verify().tolist() == [0]


def _gpu_count():
    try:
        out = subprocess.run(["nvidia-smi", "-L"], capture_output=True, text=True, timeout=20).stdout
        return sum(1 for ln in out.splitlines() if ln.startswith("GPU "))
    except Exception:
        return 0


@pytest.mark.skipif(_gpu_count() < 2, reason="needs >= 2 GPUs (one rank per GPU)")
def test_two_rank_sharded_calls_over_nccl(tmp_path):
    """Two processes, one GPU each, NO torch: the library's own communicator (id handed over through a file), then the
    sharded state root and the sharded verify batch must agree with the single-GPU answers on both ranks."""
    worker = ROOT / "tests" / "mp_sharded_worker.py"
    procs = []
    for r in range(2):
        env = dict(os.environ, B200_TEST_RANK=str(r), B200_TEST_WORLD="2", B200_TEST_DIR=str(tmp_path), CUDA_VISIBLE_DEVICES=str(r))
        procs.append(subprocess.Popen([sys.executable, str(worker)], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=900)[0] for p in procs]
    for r, (p, o) in enumerate(zip(procs, outs)):
        assert p.returncode == 0, f"rank {r}:\n{o}"
        assert "SHARDED_OK" in o, o
