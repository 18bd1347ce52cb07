"""deneb process_epoch / process_slots on the device-resident state against the CPU oracle (oracle/epoch_oracle.py)
and the golden file (tests/golden/epoch_cases.json)."""
import ctypes as C
import hashlib
import json
from pathlib import Path

import numpy as np
import pytest

from ethereum_consensus_b200 import _lib, epoch, ssz
from ethereum_consensus_b200 import state as S
from oracle import epoch_oracle as eo
from tests.golden import make_epoch_golden as mk

pytestmark = pytest.mark.gpu
GOLDEN = json.loads((Path(__file__).resolve().parent / "golden" / "epoch_cases.json").read_text())["cases"]


def _ids(c):
    return f"{c['preset']}-{c['name']}"


def _upload(st):
    return ssz.DeviceBeaconState(S.serialize(st), st.preset)


def _refused(dev):
    out = (C.c_uint8 * 32)()
    L = _lib.lib()
    n = C.c_size_t(0)
    return (L.b200_state_root(dev._h, out) == _lib.ERR_BAD_ARG and L.b200_state_root_incremental(dev._h, out) == _lib.ERR_BAD_ARG
            and L.b200_state_serialized_len(dev._h, C.byref(n)) == _lib.ERR_BAD_ARG
            and L.b200_state_process_epoch_deneb(dev._h, epoch.ALL) == _lib.ERR_BAD_ARG)


@pytest.mark.parametrize("case", GOLDEN, ids=_ids)
def test_golden_process_epoch(engine, case):
    pre = mk.build_state(case["name"], case["preset"], case["seed"])
    dev = _upload(pre)
    rc = _lib.lib().b200_state_process_epoch_deneb(dev._h, epoch.ALL)
    assert rc == case["code"]
    if rc:
        assert _refused(dev)
        return
    post = dev.to_ssz()
    assert hashlib.sha256(post.tobytes()).hexdigest() == case["post_ssz_sha256"]
    assert dev.hash_tree_root_incremental().hex() == case["post_root"]
    assert dev.hash_tree_root().hex() == case["post_root"]


@pytest.mark.parametrize("case", [c for c in GOLDEN if c["code"] == 0 or c["preset"] == "minimal"], ids=_ids)
def test_each_stage_alone(engine, case):
    for bit in range(12):
        code, want = mk.run_case(case["name"], case["preset"], case["seed"], eo.process_epoch_numpy, 1 << bit)
        dev = _upload(mk.build_state(case["name"], case["preset"], case["seed"]))
        rc = _lib.lib().b200_state_process_epoch_deneb(dev._h, 1 << bit)
        assert rc == code, eo.STAGES[bit]
        if rc == 0:
            assert dev.to_ssz().tobytes() == S.serialize(want).tobytes(), eo.STAGES[bit]
            assert dev.hash_tree_root_incremental() == eo.state_root(want), eo.STAGES[bit]
        dev.close()


def test_python_errors(engine):
    dev = _upload(mk.build_state("overflow", "minimal", 1))
    with pytest.raises(epoch.StateTransitionInvalid):
        epoch.process_epoch(dev)
    with pytest.raises(_lib.EngineError):
        dev.hash_tree_root()
    dev = _upload(mk.build_state("invalid_sync_key", "minimal", 1))
    from ethereum_consensus_b200 import crypto
    with pytest.raises(crypto.BLSTError):
        epoch.process_epoch(dev)
    dev = _upload(mk.build_state("genesis", "minimal", 1))
    with pytest.raises(epoch.TransitionToPreviousSlot):
        epoch.process_slots(dev, 7)
    epoch.process_slots(dev, 8)   # still usable: a refused slot changes nothing


def test_edge_handles(engine):
    st = mk.build_state("genesis", "minimal", 2)
    st.validators = st.validators[:0]
    st.balances = st.balances[:0]
    st.previous_epoch_participation = st.previous_epoch_participation[:0]
    st.current_epoch_participation = st.current_epoch_participation[:0]
    st.inactivity_scores = st.inactivity_scores[:0]
    dev = _upload(st)
    L = _lib.lib()
    assert L.b200_state_process_epoch_deneb(dev._h, epoch.ALL) == _lib.ERR_BAD_ARG
    assert L.b200_state_process_slots_deneb(dev._h, 10**6) == _lib.ERR_BAD_ARG
    assert dev.to_ssz().tobytes() == S.serialize(st).tobytes()   # n = 0 still downloads
    st = mk.build_state("genesis", "minimal", 2)
    st.inactivity_scores = st.inactivity_scores[:-1]   # a list shorter than the registry
    dev = _upload(st)
    assert L.b200_state_process_epoch_deneb(dev._h, epoch.ALL) == _lib.ERR_BAD_ARG
    assert L.b200_state_process_epoch_deneb(None, epoch.ALL) == _lib.ERR_BAD_ARG
    dev = _upload(mk.build_state("genesis", "minimal", 2))
    assert L.b200_state_process_epoch_deneb(dev._h, 1 << 12) == _lib.ERR_BAD_ARG


def test_sharded_handle_refused(engine):
    from ethereum_consensus_b200 import parallel
    parallel.comm_init(0, 1)
    st = mk.build_state("genesis", "minimal", 2)
    dev = ssz.DeviceBeaconState(S.serialize(st), "minimal", sharded=True)
    L = _lib.lib()
    n = C.c_size_t(0)
    assert L.b200_state_process_epoch_deneb(dev._h, epoch.ALL) == _lib.ERR_BAD_ARG
    assert L.b200_state_process_slots_deneb(dev._h, 100) == _lib.ERR_BAD_ARG
    assert L.b200_state_serialized_len(dev._h, C.byref(n)) == _lib.ERR_BAD_ARG


def test_mainnet_2p20_one_epoch_matches_numpy_oracle(engine):
    """config-3 scale: 2**20 validators, mainnet preset, one process_epoch byte-exact against the numpy form."""
    n = 1 << 20
    st = mk.base_state("mainnet", n, mk.plain_epoch("mainnet", 269_500), 0xB200)
    rng = np.random.default_rng(7)
    v = st.validators
    v["effective_balance"] = (rng.integers(15, 33, n) * 10**9).astype(np.uint64)
    v["slashed"] = rng.integers(0, 512, n) == 0
    v["withdrawable_epoch"] = np.where(v["slashed"], 269_500 + 4096, S.FAR_FUTURE_EPOCH)
    v["exit_epoch"] = np.where(v["slashed"], 269_505, S.FAR_FUTURE_EPOCH)
    pend = rng.integers(0, 2000, n) == 0
    v["activation_epoch"] = np.where(pend, S.FAR_FUTURE_EPOCH, 0)
    v["activation_eligibility_epoch"] = np.where(pend, rng.integers(0, 269_000, n), 0)
    st.slashings[::7] = 10**9
    st.balances = (v["effective_balance"] + rng.integers(0, 2 * 10**9, n)).astype("<u8")
    dev = _upload(st)
    epoch.process_epoch(dev)
    assert eo.process_epoch_numpy(st) == 0
    assert dev.to_ssz().tobytes() == S.serialize(st).tobytes()
    assert dev.hash_tree_root_incremental() == dev.hash_tree_root()


def test_process_slots_ten_epochs_minimal(engine):
    """process_slots across ten epochs with block-like writes in between; crosses an eth1 period and a
    sync-committee / historical-summaries boundary; after every epoch the device state equals the oracle's."""
    C_ = eo.CONSTS["minimal"]
    spe = C_["SLOTS_PER_EPOCH"]
    st = mk.base_state("minimal", 64, 30, 0x5107, real_keys=True)   # epochs 31..40 cross 31->32 (sync, eth1) and 35->36
    dev = _upload(st)
    rng = np.random.default_rng(3)
    slot = int.from_bytes(st.fixed["slot"], "little")
    for k in range(10):
        idx = np.sort(rng.choice(64, 16, replace=False)).astype(np.uint64)
        flags = rng.integers(0, 8, 16, dtype=np.uint8)
        bal = (32 * 10**9 + rng.integers(-10**9, 10**9, 16)).astype("<u8")
        dev.update_elements("current_epoch_participation", idx, flags)
        dev.update_elements("balances", idx, bal)
        st.current_epoch_participation[idx] = flags
        st.balances[idx] = bal
        slot += spe
        epoch.process_slots(dev, slot)
        assert eo.process_slots(st, slot) == 0
        assert dev.to_ssz().tobytes() == S.serialize(st).tobytes(), k
        assert dev.hash_tree_root_incremental() == eo.state_root(st), k


def _device_apply(pre, preset, bit):
    dev = ssz.DeviceBeaconState(np.frombuffer(pre, np.uint8), preset)
    try:
        if _lib.lib().b200_state_process_epoch_deneb(dev._h, bit) != 0:
            return None
        return dev.to_ssz().tobytes()
    finally:
        dev.close()


def test_epoch_runner_on_synthetic_tree_device(engine, tmp_path):
    from tests import spec_vectors as sv
    from tests import spec_vectors_epoch as sve
    picks = [(c["name"], c["preset"], c["seed"], mk.build_state) for c in GOLDEN
             if c["name"] in ("genesis_plus_1", "ejection_churn", "sync_and_historical", "overflow", "eth1_period")]
    base = sve.synthetic_tree(tmp_path / "consensus-spec-tests", picks)
    n = 0
    for config, fork, handler, case in sv.walk(base, "epoch_processing", sve.EPOCH_HANDLERS):
        ok, why = sve.run_epoch_case(config, handler, case, _device_apply)
        assert ok, (config, handler, case.name, why)
        n += 1
    assert n == len(picks) * 12


@pytest.mark.skipif(__import__("tests.spec_vectors", fromlist=["x"]).vectors_root() is None,
                    reason="consensus-spec-tests not present (offline); set CONSENSUS_SPEC_TESTS")
def test_epoch_runner_on_real_vectors(engine):
    from tests import spec_vectors as sv
    from tests import spec_vectors_epoch as sve
    for config, fork, handler, case in sv.walk(sv.vectors_root(), "epoch_processing", sve.EPOCH_HANDLERS):
        if fork != "deneb":
            continue
        for apply in (sve.oracle_apply, _device_apply):
            ok, why = sve.run_epoch_case(config, handler, case, apply)
            assert ok, (config, handler, case.name, why)
