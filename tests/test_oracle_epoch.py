"""CPU checks of the epoch-processing oracle (oracle/epoch_oracle.py), its golden file and constants, and the build of
epoch.cu for sm_100a."""
import json
import os
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from ethereum_consensus_b200 import state as S
from oracle import epoch_oracle as eo
from tests.golden import make_epoch_golden as mk

ROOT = Path(__file__).resolve().parent.parent
GOLDEN = json.loads((ROOT / "tests" / "golden" / "epoch_cases.json").read_text())
CONSTANTS = json.loads((ROOT / "tests" / "golden" / "epoch_constants.json").read_text())
# the reference's source tree (ethereum-consensus/src), when it is available next to the checkout
REF_SRC = Path(os.environ.get("B200_REFERENCE_SRC", "/root/reference/ethereum-consensus/src"))


def _ids(c):
    return f"{c['preset']}-{c['name']}"


@pytest.mark.parametrize("case", GOLDEN["cases"], ids=_ids)
def test_literal_and_numpy_forms_agree(case):
    a_code, a = mk.run_case(case["name"], case["preset"], case["seed"], eo.process_epoch_literal)
    b_code, b = mk.run_case(case["name"], case["preset"], case["seed"], eo.process_epoch_numpy)
    assert a_code == b_code == case["code"]
    if a_code == 0:
        assert S.serialize(a).tobytes() == S.serialize(b).tobytes()


@pytest.mark.parametrize("case", [c for c in GOLDEN["cases"] if c["preset"] == "minimal"], ids=_ids)
def test_forms_agree_stage_by_stage(case):
    for bit in range(12):
        a_code, a = mk.run_case(case["name"], case["preset"], case["seed"], eo.process_epoch_literal, 1 << bit)
        b_code, b = mk.run_case(case["name"], case["preset"], case["seed"], eo.process_epoch_numpy, 1 << bit)
        assert a_code == b_code, eo.STAGES[bit]
        if a_code == 0:
            assert S.serialize(a).tobytes() == S.serialize(b).tobytes(), eo.STAGES[bit]


def test_golden_regenerates_byte_for_byte():
    assert mk.render() == (ROOT / "tests" / "golden" / "epoch_cases.json").read_text()


def test_golden_covers_the_edges():
    by = {(c["preset"], c["name"]): c for c in GOLDEN["cases"]}
    for preset in ("minimal", "mainnet"):
        assert by[(preset, "overflow")]["code"] == eo.INVALID
        assert 1 <= by[(preset, "invalid_sync_key")]["code"] <= 7
    # the boundary scenarios really cross their boundaries
    C = eo.CONSTS["minimal"]
    code, st = mk.run_case("sync_and_historical", "minimal", by[("minimal", "sync_and_historical")]["seed"])
    pre = mk.build_state("sync_and_historical", "minimal", by[("minimal", "sync_and_historical")]["seed"])
    assert len(st.historical_summaries) == len(pre.historical_summaries) + 1
    assert st.current_sync_committee == pre.next_sync_committee and st.next_sync_committee != pre.next_sync_committee
    code, st = mk.run_case("eth1_period", "minimal", by[("minimal", "eth1_period")]["seed"])
    assert len(st.eth1_data_votes) == 0 and C["EPOCHS_PER_ETH1_VOTING_PERIOD"] == 4
    code, st = mk.run_case("balance_saturates", "minimal", by[("minimal", "balance_saturates")]["seed"])
    assert int((st.balances == 0).sum()) > 0
    code, st = mk.run_case("finality_rule_234", "minimal", by[("minimal", "finality_rule_234")]["seed"])
    pre = mk.build_state("finality_rule_234", "minimal", by[("minimal", "finality_rule_234")]["seed"])
    assert st.fixed["finalized_checkpoint"] == pre.fixed["previous_justified_checkpoint"]


def test_ejections_respect_the_churn():
    code, st = mk.run_case("ejection_churn", "minimal", 1)
    C = eo.CONSTS["minimal"]
    exits = st.validators["exit_epoch"][st.validators["exit_epoch"] != S.FAR_FUTURE_EPOCH]
    _, counts = np.unique(exits, return_counts=True)
    assert counts.max() <= C["MIN_PER_EPOCH_CHURN_LIMIT"] and len(counts) >= 3


def test_constants_match_the_fixture():
    for preset in ("mainnet", "minimal"):
        for name, value in CONSTANTS[preset].items():
            assert eo.CONSTS[preset][name] == value, (preset, name)
    # the CUDA table (epoch.cu) holds the same values
    src = (ROOT / "ethereum_consensus_b200" / "csrc" / "epoch.cu").read_text()
    for name in ["EFFECTIVE_BALANCE_INCREMENT", "MAX_EFFECTIVE_BALANCE", "EJECTION_BALANCE", "BASE_REWARD_FACTOR",
                 "HYSTERESIS_QUOTIENT", "HYSTERESIS_DOWNWARD_MULTIPLIER", "HYSTERESIS_UPWARD_MULTIPLIER", "MIN_SEED_LOOKAHEAD",
                 "MAX_SEED_LOOKAHEAD", "MIN_EPOCHS_TO_INACTIVITY_PENALTY", "INACTIVITY_PENALTY_QUOTIENT_BELLATRIX",
                 "PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX", "INACTIVITY_SCORE_BIAS", "INACTIVITY_SCORE_RECOVERY_RATE",
                 "MIN_VALIDATOR_WITHDRAWABILITY_DELAY"]:
        m = re.search(rf"\b{name} = (\d+)", src)
        assert m and int(m.group(1)) == CONSTANTS["mainnet"][name] == CONSTANTS["minimal"][name], name
    fields = ["SLOTS_PER_EPOCH", "SLOTS_PER_HISTORICAL_ROOT", "EPOCHS_PER_HISTORICAL_VECTOR", "EPOCHS_PER_SLASHINGS_VECTOR",
              "SYNC_COMMITTEE_SIZE", "EPOCHS_PER_SYNC_COMMITTEE_PERIOD", "EPOCHS_PER_ETH1_VOTING_PERIOD", "SHUFFLE_ROUND_COUNT",
              "MIN_PER_EPOCH_CHURN_LIMIT", "MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT", "CHURN_LIMIT_QUOTIENT", "HISTORICAL_ROOTS_LIMIT"]
    for preset in ("mainnet", "minimal"):
        row = re.search(r"\{([^{}]*)\},\s*// " + preset, src).group(1)
        vals = [int(eval(x.replace("ull", ""))) for x in row.split(",")]  # noqa: S307 - integer literals from our source
        assert vals == [CONSTANTS[preset][f] for f in fields], preset


@pytest.mark.skipif(not REF_SRC.is_dir(), reason="the reference source tree is not available")
def test_constant_fixture_matches_the_reference_files():
    assert mk.reference_constants(REF_SRC) == CONSTANTS


def test_process_slots_oracle_crosses_an_epoch():
    st = mk.build_state("inactivity_leak", "minimal", 5)
    s0 = int.from_bytes(st.fixed["slot"], "little")
    assert eo.process_slots(st, s0 + 2) == 0
    assert int.from_bytes(st.fixed["slot"], "little") == s0 + 2
    with pytest.raises(ValueError):
        eo.process_slots(st, s0)


def test_ssz_round_trip():
    st = mk.build_state("eth1_period", "mainnet", 3)
    b = S.serialize(st).tobytes()
    assert S.serialize(eo.from_ssz(b, "mainnet")).tobytes() == b


def test_epoch_cu_builds_without_spills(tmp_path):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    if not Path(nvcc).exists():
        pytest.skip("nvcc not available")
    r = subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "--expt-relaxed-constexpr",
                        "-Xptxas", "-v", "-c", str(ROOT / "ethereum_consensus_b200" / "csrc" / "epoch.cu"), "-o",
                        str(tmp_path / "epoch.o")], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    spills = re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", r.stderr)
    assert spills and all(a == "0" and b == "0" for a, b in spills)


def test_epoch_runner_on_synthetic_tree(tmp_path):
    from tests import spec_vectors as sv
    from tests import spec_vectors_epoch as sve
    picks = [(c["name"], c["preset"], c["seed"], mk.build_state) for c in GOLDEN["cases"]
             if c["preset"] == "minimal" and c["name"] in ("genesis_plus_1", "ejection_churn", "sync_and_historical", "overflow")]
    base = sve.synthetic_tree(tmp_path / "consensus-spec-tests", picks)
    n = 0
    for config, fork, handler, case in sv.walk(base, "epoch_processing", sve.EPOCH_HANDLERS):
        ok, why = sve.run_epoch_case(config, handler, case, sve.oracle_apply)
        assert ok, (handler, case.name, why)
        n += 1
    assert n == len(picks) * 12
    assert not (base / "tests/minimal/deneb/epoch_processing/inactivity_updates/pyspec_tests/overflow/post.ssz_snappy").exists()
