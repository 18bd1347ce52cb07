"""Writes tests/golden/epoch_cases.json: deneb process_epoch scenarios for both presets at small N.

Each case is rebuilt from its name, preset and seed by `build_state` (deterministic), so the file only holds the
scenario parameters, the return code, the SHA-256 of the post-state SSZ and the post-state root (hashlib oracle).
Post-states come from the numpy form of oracle/epoch_oracle.py; tests/test_oracle_epoch.py checks that the literal
form agrees on every case and that this script reproduces the file byte for byte.

    python tests/golden/make_epoch_golden.py
"""
from __future__ import annotations

import hashlib
import json
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[2]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

from ethereum_consensus_b200 import state as S  # noqa: E402
from oracle import bls_oracle as bo  # noqa: E402
from oracle import epoch_oracle as eo  # noqa: E402

OUT = Path(__file__).resolve().parent / "epoch_cases.json"
N = 64
FF = S.FAR_FUTURE_EPOCH
GWEI = 10**9
SCENARIOS = ["genesis", "genesis_plus_1", "finality_rule_234", "finality_rule_23", "finality_rule_123", "finality_rule_12",
             "inactivity_leak", "balance_saturates", "ejection_churn", "activation_queue", "slashings_midpoint",
             "hysteresis_edges", "eth1_period", "sync_and_historical", "overflow", "invalid_sync_key"]


def _cp(epoch: int, tag: bytes) -> bytes:
    return int(epoch).to_bytes(8, "little") + hashlib.sha256(tag).digest()


def boundary_epoch(preset: str, kind: str, base: int = 40) -> int:
    C = eo.CONSTS[preset]
    period = {"eth1": C["EPOCHS_PER_ETH1_VOTING_PERIOD"], "sync": C["EPOCHS_PER_SYNC_COMMITTEE_PERIOD"]}[kind]
    e = base
    while (e + 1) % period:
        e += 1
    if kind == "eth1":   # keep clear of the sync / historical boundary
        while (e + 1) % C["EPOCHS_PER_SYNC_COMMITTEE_PERIOD"] == 0 or (e + 1) % (C["SLOTS_PER_HISTORICAL_ROOT"] // C["SLOTS_PER_EPOCH"]) == 0:
            e += period
    return e


def plain_epoch(preset: str, e: int) -> int:
    """the first epoch >= e whose end crosses none of the period boundaries"""
    C = eo.CONSTS[preset]
    periods = [C["EPOCHS_PER_ETH1_VOTING_PERIOD"], C["EPOCHS_PER_SYNC_COMMITTEE_PERIOD"],
               C["SLOTS_PER_HISTORICAL_ROOT"] // C["SLOTS_PER_EPOCH"]]
    while any((e + 1) % p == 0 for p in periods):
        e += 1
    return e


def base_state(preset: str, n: int, epoch: int, seed: int, real_keys: bool = False) -> S.SynthState:
    """A consistent deneb state at the last slot of `epoch`: every validator active since genesis, justified and
    finalized checkpoints at the usual distance, random participation."""
    C = eo.CONSTS[preset]
    pks = np.frombuffer(b"".join(bo.sk_to_pk(1000 + i) for i in range(n)), np.uint8).reshape(n, 48) if real_keys else None
    st = S.synth_state(n, preset, seed=seed, n_historical_summaries=2, n_historical_roots=1, pubkeys=pks)
    rng = np.random.default_rng(seed)
    v = st.validators
    v["effective_balance"] = 32 * GWEI
    v["slashed"] = 0
    v["activation_eligibility_epoch"] = 0
    v["activation_epoch"] = 0
    v["exit_epoch"] = FF
    v["withdrawable_epoch"] = FF
    st.balances = (32 * GWEI + rng.integers(-10**8, 10**8, n)).astype("<u8")
    st.previous_epoch_participation = rng.integers(0, 8, n, dtype=np.uint8)
    st.current_epoch_participation = rng.integers(0, 8, n, dtype=np.uint8)
    st.inactivity_scores = rng.integers(0, 40, n).astype("<u8")
    st.slashings = np.zeros(C["EPOCHS_PER_SLASHINGS_VECTOR"], "<u8")
    f = st.fixed
    f["slot"] = int(epoch * C["SLOTS_PER_EPOCH"] + C["SLOTS_PER_EPOCH"] - 1).to_bytes(8, "little")
    f["justification_bits"] = bytes([0b0011])
    f["previous_justified_checkpoint"] = _cp(max(0, epoch - 2), b"pj")
    f["current_justified_checkpoint"] = _cp(max(0, epoch - 1), b"cj")
    f["finalized_checkpoint"] = _cp(max(0, epoch - 2), b"fin")
    return st


def build_state(name: str, preset: str, seed: int) -> S.SynthState:
    C = eo.CONSTS[preset]
    e = plain_epoch(preset, 40)
    if name == "genesis":
        return base_state(preset, N, 0, seed)
    if name == "genesis_plus_1":
        return base_state(preset, N, 1, seed)
    if name.startswith("finality_rule"):
        st = base_state(preset, N, e, seed)
        full, none = np.full(N, 7, np.uint8), np.zeros(N, np.uint8)
        f = st.fixed
        st.previous_epoch_participation = full
        st.current_epoch_participation = none
        if name == "finality_rule_234":
            f["justification_bits"] = bytes([0b0111]); f["previous_justified_checkpoint"] = _cp(e - 3, b"pj")
        elif name == "finality_rule_23":
            f["justification_bits"] = bytes([0b0001]); f["previous_justified_checkpoint"] = _cp(e - 2, b"pj")
        elif name == "finality_rule_123":
            st.current_epoch_participation = full
            f["justification_bits"] = bytes([0b0011]); f["current_justified_checkpoint"] = _cp(e - 2, b"cj")
            f["previous_justified_checkpoint"] = _cp(e - 5, b"pj")
        else:
            st.current_epoch_participation = full
            f["justification_bits"] = bytes([0b0001]); f["current_justified_checkpoint"] = _cp(e - 1, b"cj")
            f["previous_justified_checkpoint"] = _cp(e - 5, b"pj")
        return st
    if name == "inactivity_leak":
        st = base_state(preset, N, e, seed)
        st.fixed["finalized_checkpoint"] = _cp(e - 10, b"fin")
        return st
    if name == "balance_saturates":
        st = base_state(preset, N, e, seed)
        st.fixed["finalized_checkpoint"] = _cp(e - 10, b"fin")
        st.previous_epoch_participation[: N // 2] = 0
        st.balances[: N // 2] = np.arange(N // 2, dtype=np.uint64) * 1000
        st.inactivity_scores[: N // 2] = 10**6
        return st
    if name == "ejection_churn":
        st = base_state(preset, N, e, seed)
        v = st.validators
        v["effective_balance"][: 3 * C["MIN_PER_EPOCH_CHURN_LIMIT"] + 1] = 16 * GWEI
        v["effective_balance"][5] = 17 * GWEI   # above the ejection balance
        aee_epoch = e + 1 + C["MAX_SEED_LOOKAHEAD"]
        v["exit_epoch"][N - 2:] = aee_epoch     # the queue epoch already holds two exits
        v["withdrawable_epoch"][N - 2:] = aee_epoch + 256
        return st
    if name == "activation_queue":
        st = base_state(preset, N, e, seed)
        v = st.validators
        k = 3 * C["MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT"]
        v["activation_epoch"][10:10 + k] = FF
        v["activation_eligibility_epoch"][10:10 + k] = np.array([e - 5 + (i % 3) for i in range(k)][::-1], np.uint64)
        v["activation_eligibility_epoch"][40] = e + 3   # above the finalized epoch: waits
        v["activation_epoch"][40] = FF
        v["activation_eligibility_epoch"][41] = FF      # not yet queued, at MAX_EFFECTIVE_BALANCE: becomes eligible
        v["activation_epoch"][41] = FF
        return st
    if name == "slashings_midpoint":
        st = base_state(preset, N, e, seed)
        v = st.validators
        half = C["EPOCHS_PER_SLASHINGS_VECTOR"] // 2
        v["slashed"][:6] = 1
        v["exit_epoch"][:6] = e + 2
        v["withdrawable_epoch"][:6] = [e + half, e + half, e + half - 1, e + half + 1, e + half, e + half]
        v["effective_balance"][1] = 31 * GWEI
        st.slashings[::3] = 5 * GWEI
        return st
    if name == "hysteresis_edges":
        st = base_state(preset, N, e, seed)
        st.previous_epoch_participation[:] = 7
        st.current_epoch_participation[:] = 7
        v = st.validators
        q = GWEI // 4
        v["effective_balance"][:8] = 20 * GWEI
        # down edge: balance + 0.25 < eb updates, == does not; up edge: eb + 1.25 < balance updates, == does not
        st.balances[:8] = [20 * GWEI - q - 1, 20 * GWEI - q, 20 * GWEI + 5 * q + 1, 20 * GWEI + 5 * q,
                           40 * GWEI, 0, 33 * GWEI + 7, 20 * GWEI - q - 10**6]
        st.inactivity_scores[:] = 0
        return st
    if name == "eth1_period":
        return base_state(preset, N, boundary_epoch(preset, "eth1"), seed)
    if name == "sync_and_historical":
        return base_state(preset, N, boundary_epoch(preset, "sync"), seed, real_keys=True)
    if name == "overflow":
        st = base_state(preset, N, e, seed)
        st.previous_epoch_participation[3] = 0
        st.inactivity_scores[3] = (1 << 64) - 2
        return st
    if name == "invalid_sync_key":
        st = base_state(preset, N, boundary_epoch(preset, "sync"), seed)
        st.validators["public_key"] = np.zeros((N, 48), np.uint8).view("V48").reshape(N)   # no compression flag
        return st
    raise KeyError(name)


def run_case(name: str, preset: str, seed: int, form=eo.process_epoch_numpy, mask: int = eo.ALL):
    st = build_state(name, preset, seed)
    code = form(st, mask)
    return code, st


def case_record(name: str, preset: str, seed: int) -> dict:
    code, st = run_case(name, preset, seed)
    rec = {"name": name, "preset": preset, "seed": seed, "n": N, "code": code}
    if code == 0:
        rec["post_ssz_sha256"] = hashlib.sha256(S.serialize(st).tobytes()).hexdigest()
        rec["post_root"] = eo.state_root(st).hex()
    return rec


def cases() -> list:
    return [case_record(name, preset, 0xE90C + k) for preset in ("minimal", "mainnet") for k, name in enumerate(SCENARIOS)]


def render() -> str:
    return json.dumps({"n": N, "cases": cases()}, indent=1, sort_keys=True) + "\n"


if __name__ == "__main__":
    OUT.write_text(render())
    print(f"wrote {OUT}")


# ---- constants: extracted from the reference's preset and config files into epoch_constants.json (a data fixture)
CONST_FILES = {  # name -> file under ethereum-consensus/src/ holding `pub const NAME: T = value;` for each preset
    **{k: "phase0/presets/{p}.rs" for k in ["EFFECTIVE_BALANCE_INCREMENT", "MAX_EFFECTIVE_BALANCE", "BASE_REWARD_FACTOR",
                                           "HYSTERESIS_QUOTIENT", "HYSTERESIS_DOWNWARD_MULTIPLIER", "HYSTERESIS_UPWARD_MULTIPLIER",
                                           "MIN_SEED_LOOKAHEAD", "MAX_SEED_LOOKAHEAD", "MIN_EPOCHS_TO_INACTIVITY_PENALTY",
                                           "SLOTS_PER_EPOCH", "EPOCHS_PER_ETH1_VOTING_PERIOD", "SHUFFLE_ROUND_COUNT",
                                           "SLOTS_PER_HISTORICAL_ROOT", "EPOCHS_PER_HISTORICAL_VECTOR", "EPOCHS_PER_SLASHINGS_VECTOR",
                                           "HISTORICAL_ROOTS_LIMIT"]},
    **{k: "altair/presets/{p}.rs" for k in ["EPOCHS_PER_SYNC_COMMITTEE_PERIOD", "SYNC_COMMITTEE_SIZE"]},
    **{k: "bellatrix/presets/{p}.rs" for k in ["INACTIVITY_PENALTY_QUOTIENT_BELLATRIX", "PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX"]},
    **{k: "configs/{p}.rs" for k in ["EJECTION_BALANCE", "MIN_PER_EPOCH_CHURN_LIMIT", "MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT",
                                     "CHURN_LIMIT_QUOTIENT", "INACTIVITY_SCORE_BIAS", "INACTIVITY_SCORE_RECOVERY_RATE",
                                     "MIN_VALIDATOR_WITHDRAWABILITY_DELAY"]},
}
CONST_OUT = Path(__file__).resolve().parent / "epoch_constants.json"


def reference_constants(src: Path) -> dict:
    """{preset: {name: value}} read from `pub const NAME: T = <expr>;` lines (expr: integers, `_`, `*`, `10u64.pow(k)`)."""
    import re
    out = {}
    for p in ("mainnet", "minimal"):
        d = {}
        for name, rel in CONST_FILES.items():
            text = (src / rel.format(p=p)).read_text()
            m = re.search(rf"pub const {name}: [\w]+ = ([^;]+);", text)
            if m is None:
                raise KeyError(f"{name} not in {rel.format(p=p)}")
            expr = re.sub(r"(\d+)u64\.pow\((\d+)\)", r"\1**\2", m.group(1).replace("_", ""))
            if not re.fullmatch(r"[\d\s*()+-]+", expr):
                raise ValueError(f"{name}: unexpected expression {m.group(1)!r}")
            d[name] = int(eval(expr))  # noqa: S307 - digits and operators only (checked above)
        out[p] = d
    return out
