"""CPU oracle for deneb `process_epoch` / `process_slots` — TEST INFRASTRUCTURE ONLY.

The spec (/root/reference/ethereum-consensus/src/deneb/spec/mod.rs:965-1004, deneb/epoch_processing.rs:11) restated in
two forms over `state.SynthState`:
  * `process_epoch_literal` — function by function over Python ints (small N): get_flag_index_deltas and
    get_inactivity_penalty_deltas build their delta lists and apply them pair by pair, initiate_validator_exit rescans
    the registry.  Only `get_total_active_balance` is hoisted (it has the same value throughout stages 0..4), so that
    rewards cost O(N) instead of O(N^2).
  * `process_epoch_numpy` — vectorised uint64 work with explicit overflow checks, fast enough for 2**20 validators.
The host-only stages (justification weighing, eth1 / slashings / randao resets, historical summaries, sync-committee
selection) are shared: they are a few lines of scalar logic with no per-validator work.
Any uint64 overflow, and every spec assertion, is an invalid transition: `INVALID` (18).  An invalid key in the next
sync committee returns its blst code (bls_oracle.eth_aggregate_public_keys).
"""
from __future__ import annotations

import copy
import hashlib
import struct
from typing import Dict, List, Tuple

import numpy as np

from ethereum_consensus_b200.state import PRESETS, VALIDATOR_DTYPE, SynthState, FAR_FUTURE_EPOCH
from oracle import bls_oracle as bo
from oracle import shuffle_oracle as sh
from oracle import ssz_oracle as so

INVALID = 18
U64 = (1 << 64) - 1
ALL = 0xFFF
STAGES = ["justification_and_finalization", "inactivity_updates", "rewards_and_penalties", "registry_updates",
          "slashings", "eth1_data_reset", "effective_balance_updates", "slashings_reset", "randao_mixes_reset",
          "historical_summaries_update", "participation_flag_updates", "sync_committee_updates"]

# phase0/presets/*.rs, altair/presets/*.rs, bellatrix/presets/*.rs, configs/*.rs (pinned by tests/test_oracle_epoch.py)
COMMON = dict(EFFECTIVE_BALANCE_INCREMENT=10**9, MAX_EFFECTIVE_BALANCE=32 * 10**9, EJECTION_BALANCE=16 * 10**9,
              BASE_REWARD_FACTOR=64, HYSTERESIS_QUOTIENT=4, HYSTERESIS_DOWNWARD_MULTIPLIER=1, HYSTERESIS_UPWARD_MULTIPLIER=5,
              MIN_SEED_LOOKAHEAD=1, MAX_SEED_LOOKAHEAD=4, MIN_EPOCHS_TO_INACTIVITY_PENALTY=4,
              INACTIVITY_PENALTY_QUOTIENT_BELLATRIX=16_777_216, PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX=3,
              INACTIVITY_SCORE_BIAS=4, INACTIVITY_SCORE_RECOVERY_RATE=16, MIN_VALIDATOR_WITHDRAWABILITY_DELAY=256)
CONSTS: Dict[str, Dict[str, int]] = {
    "mainnet": dict(COMMON, SLOTS_PER_EPOCH=32, EPOCHS_PER_SYNC_COMMITTEE_PERIOD=256, EPOCHS_PER_ETH1_VOTING_PERIOD=64,
                    SHUFFLE_ROUND_COUNT=90, MIN_PER_EPOCH_CHURN_LIMIT=4, MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT=8,
                    CHURN_LIMIT_QUOTIENT=65536, **PRESETS["mainnet"]),
    "minimal": dict(COMMON, SLOTS_PER_EPOCH=8, EPOCHS_PER_SYNC_COMMITTEE_PERIOD=8, EPOCHS_PER_ETH1_VOTING_PERIOD=4,
                    SHUFFLE_ROUND_COUNT=10, MIN_PER_EPOCH_CHURN_LIMIT=2, MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT=4,
                    CHURN_LIMIT_QUOTIENT=32, **PRESETS["minimal"]),
}
WEIGHTS = (14, 26, 14)   # TIMELY_SOURCE, TIMELY_TARGET, TIMELY_HEAD
WEIGHT_DENOMINATOR = 64


class Invalid(Exception):
    pass


def _u64(b: bytes) -> int:
    return int.from_bytes(b[:8], "little")


def _p64(x: int) -> bytes:
    return int(x).to_bytes(8, "little")


def _check(x: int, what: str) -> int:
    if x > U64 or x < 0:
        raise Invalid(what)
    return x


def integer_squareroot(n: int) -> int:
    x = n
    y = (x + 1) // 2
    while y < x:
        x = y
        y = (x + n // x) // 2
    return x


# ------------------------------------------------------------------------------------------------ SSZ <-> SynthState

def from_ssz(buf, preset: str) -> SynthState:
    """Parse a deneb BeaconState serialization (the inverse of state.serialize)."""
    b = bytes(buf)
    P = PRESETS[preset]
    st = SynthState(preset=preset)
    o = 0

    def take(n):
        nonlocal o
        r = b[o:o + n]
        o += n
        return r
    f = st.fixed
    f["genesis_time"] = take(8); f["genesis_validators_root"] = take(32); f["slot"] = take(8); f["fork"] = take(16)
    f["latest_block_header"] = take(112)
    st.block_roots = np.frombuffer(take(32 * P["SLOTS_PER_HISTORICAL_ROOT"]), np.uint8).reshape(-1, 32).copy()
    st.state_roots = np.frombuffer(take(32 * P["SLOTS_PER_HISTORICAL_ROOT"]), np.uint8).reshape(-1, 32).copy()
    offs = [struct.unpack("<I", take(4))[0]]
    f["eth1_data"] = take(72)
    offs.append(struct.unpack("<I", take(4))[0])
    f["eth1_deposit_index"] = take(8)
    offs += list(struct.unpack("<II", take(8)))
    st.randao_mixes = np.frombuffer(take(32 * P["EPOCHS_PER_HISTORICAL_VECTOR"]), np.uint8).reshape(-1, 32).copy()
    st.slashings = np.frombuffer(take(8 * P["EPOCHS_PER_SLASHINGS_VECTOR"]), "<u8").copy()
    offs += list(struct.unpack("<II", take(8)))
    f["justification_bits"] = take(1)
    f["previous_justified_checkpoint"] = take(40); f["current_justified_checkpoint"] = take(40); f["finalized_checkpoint"] = take(40)
    offs.append(struct.unpack("<I", take(4))[0])
    sc = 48 * P["SYNC_COMMITTEE_SIZE"] + 48
    st.current_sync_committee = take(sc); st.next_sync_committee = take(sc)
    offs.append(struct.unpack("<I", take(4))[0])
    f["next_withdrawal_index"] = take(8); f["next_withdrawal_validator_index"] = take(8)
    offs.append(struct.unpack("<I", take(4))[0])
    offs.append(len(b))
    var = [b[offs[i]:offs[i + 1]] for i in range(9)]
    st.historical_roots = np.frombuffer(var[0], np.uint8).reshape(-1, 32).copy()
    st.eth1_data_votes = np.frombuffer(var[1], np.uint8).reshape(-1, 72).copy()
    st.validators = np.frombuffer(var[2], VALIDATOR_DTYPE).copy()
    st.balances = np.frombuffer(var[3], "<u8").copy()
    st.previous_epoch_participation = np.frombuffer(var[4], np.uint8).copy()
    st.current_epoch_participation = np.frombuffer(var[5], np.uint8).copy()
    st.inactivity_scores = np.frombuffer(var[6], "<u8").copy()
    st.payload_header_fixed, st.extra_data = var[7][:584], var[7][584:]
    st.historical_summaries = np.frombuffer(var[8], np.uint8).reshape(-1, 64).copy()
    return st


def state_root(st: SynthState) -> bytes:
    from ethereum_consensus_b200.state import to_oracle_value
    return so.beacon_state_type(st.preset).htr(to_oracle_value(st))


# ------------------------------------------------------------------------------------------------ shared host stages

def _epochs(st: SynthState, C) -> Tuple[int, int]:
    cur = _u64(st.fixed["slot"]) // C["SLOTS_PER_EPOCH"]
    return cur, (cur - 1 if cur > 0 else 0)


def _block_root(st: SynthState, C, epoch: int) -> bytes:
    slot, state_slot = epoch * C["SLOTS_PER_EPOCH"], _u64(st.fixed["slot"])
    if not (slot < state_slot <= slot + C["SLOTS_PER_HISTORICAL_ROOT"]):
        raise Invalid("get_block_root_at_slot")
    return st.block_roots[slot % C["SLOTS_PER_HISTORICAL_ROOT"]].tobytes()


def weigh_justification_and_finalization(st: SynthState, C, total: int, prev_target: int, cur_target: int) -> None:
    cur, prev = _epochs(st, C)
    f = st.fixed
    old_prev, old_cur = f["previous_justified_checkpoint"], f["current_justified_checkpoint"]
    f["previous_justified_checkpoint"] = old_cur
    bits = [(f["justification_bits"][0] >> i) & 1 for i in range(4)]
    bits = [0] + bits[:3]
    _check(prev_target * 3, "weigh"); _check(cur_target * 3, "weigh"); _check(total * 2, "weigh")
    if prev_target * 3 >= total * 2:
        f["current_justified_checkpoint"] = _p64(prev) + _block_root(st, C, prev)
        bits[1] = 1
    if cur_target * 3 >= total * 2:
        f["current_justified_checkpoint"] = _p64(cur) + _block_root(st, C, cur)
        bits[0] = 1
    f["justification_bits"] = bytes([sum(b << i for i, b in enumerate(bits))])
    op, oc = _u64(old_prev), _u64(old_cur)
    if all(bits[1:4]) and op + 3 == cur:
        f["finalized_checkpoint"] = old_prev
    if all(bits[1:3]) and op + 2 == cur:
        f["finalized_checkpoint"] = old_prev
    if all(bits[0:3]) and oc + 2 == cur:
        f["finalized_checkpoint"] = old_cur
    if all(bits[0:2]) and oc + 1 == cur:
        f["finalized_checkpoint"] = old_cur


def is_in_inactivity_leak(st: SynthState, C) -> bool:
    _, prev = _epochs(st, C)
    fin = _u64(st.fixed["finalized_checkpoint"])
    return _check(prev - fin, "finality delay") > C["MIN_EPOCHS_TO_INACTIVITY_PENALTY"]


def eth1_data_reset(st, C):
    cur, _ = _epochs(st, C)
    if (cur + 1) % C["EPOCHS_PER_ETH1_VOTING_PERIOD"] == 0:
        st.eth1_data_votes = np.zeros((0, 72), np.uint8)


def slashings_reset(st, C):
    cur, _ = _epochs(st, C)
    st.slashings[(cur + 1) % C["EPOCHS_PER_SLASHINGS_VECTOR"]] = 0


def randao_mixes_reset(st, C):
    cur, _ = _epochs(st, C)
    st.randao_mixes[(cur + 1) % C["EPOCHS_PER_HISTORICAL_VECTOR"]] = st.randao_mixes[cur % C["EPOCHS_PER_HISTORICAL_VECTOR"]]


def historical_summaries_update(st, C):
    cur, _ = _epochs(st, C)
    if (cur + 1) % (C["SLOTS_PER_HISTORICAL_ROOT"] // C["SLOTS_PER_EPOCH"]) == 0:
        if len(st.historical_summaries) + 1 > C["HISTORICAL_ROOTS_LIMIT"]:
            raise Invalid("historical_summaries full")
        lim = C["SLOTS_PER_HISTORICAL_ROOT"]
        br = so.merkleize_chunks([r.tobytes() for r in st.block_roots], lim)
        sr = so.merkleize_chunks([r.tobytes() for r in st.state_roots], lim)
        row = np.frombuffer(br + sr, np.uint8).reshape(1, 64)
        st.historical_summaries = np.concatenate([st.historical_summaries.reshape(-1, 64), row])


def participation_flag_updates(st, C):
    st.previous_epoch_participation = st.current_epoch_participation.copy()
    st.current_epoch_participation = np.zeros_like(st.current_epoch_participation)


def get_seed(st, C, epoch: int, domain: bytes) -> bytes:
    ehv = C["EPOCHS_PER_HISTORICAL_VECTOR"]
    mix = st.randao_mixes[(epoch + ehv - C["MIN_SEED_LOOKAHEAD"] - 1) % ehv].tobytes()
    return hashlib.sha256(domain + _p64(epoch) + mix).digest()


def get_next_sync_committee_indices(st, C) -> List[int]:
    cur, _ = _epochs(st, C)
    epoch = cur + 1
    v = st.validators
    active = [i for i in range(len(v)) if int(v["activation_epoch"][i]) <= epoch < int(v["exit_epoch"][i])]
    n = len(active)
    if n == 0:
        raise Invalid("no active validator")
    seed = get_seed(st, C, epoch, bytes([7, 0, 0, 0]))
    out, i, cache = [], 0, {}
    while len(out) < C["SYNC_COMMITTEE_SIZE"]:
        k = i % n
        if k not in cache:
            cache[k] = active[sh.compute_shuffled_index(k, n, seed, C["SHUFFLE_ROUND_COUNT"])]
        cand = cache[k]
        rnd = hashlib.sha256(seed + _p64(i // 32)).digest()[i % 32]
        eb = int(v["effective_balance"][cand])
        if _check(eb * 255, "sync sampling") >= C["MAX_EFFECTIVE_BALANCE"] * rnd:
            out.append(cand)
        i += 1
    return out


_KEYS: Dict[bytes, tuple] = {}


def eth_aggregate_public_keys(pks: List[bytes]):
    """bls_oracle.eth_aggregate_public_keys with each distinct key validated once (a committee repeats keys when the
    registry is small): the first invalid key in order decides the code, as there."""
    acc = bo.pt_inf(bo.F1)
    for b in pks:
        if b not in _KEYS:
            _KEYS[b] = bo.key_validate(b)
        code, a = _KEYS[b]
        if code:
            return code, None
        acc = bo.pt_add(bo.F1, acc, bo.pt_from_affine(bo.F1, a))
    return 0, bo.g1_compress(bo.pt_to_affine(bo.F1, acc))


def sync_committee_updates(st, C) -> int:
    cur, _ = _epochs(st, C)
    if (cur + 1) % C["EPOCHS_PER_SYNC_COMMITTEE_PERIOD"] != 0:
        return 0
    idx = get_next_sync_committee_indices(st, C)
    keys = [st.validators["public_key"][i].tobytes() for i in idx]
    code, agg = eth_aggregate_public_keys(keys)
    if code:
        return code
    st.current_sync_committee = st.next_sync_committee
    st.next_sync_committee = b"".join(keys) + agg
    return 0


# ------------------------------------------------------------------------------------------------ literal form

def _v(st, i):
    r = st.validators[i]
    return dict(eb=int(r["effective_balance"]), slashed=bool(r["slashed"]), aee=int(r["activation_eligibility_epoch"]),
                act=int(r["activation_epoch"]), exit=int(r["exit_epoch"]), wd=int(r["withdrawable_epoch"]))


def _active(v, epoch):
    return v["act"] <= epoch < v["exit"]


def _total_balance(st, indices) -> int:
    s = sum(int(st.validators["effective_balance"][i]) for i in indices)
    return max(COMMON["EFFECTIVE_BALANCE_INCREMENT"], _check(s, "total balance"))


def _unslashed_participating(st, C, flag: int, epoch: int, part) -> List[int]:
    out = []
    for i in range(len(st.validators)):
        v = _v(st, i)
        if _active(v, epoch) and not v["slashed"] and (int(part[i]) >> flag) & 1:
            out.append(i)
    return out


def _eligible(st, prev) -> List[int]:
    out = []
    for i in range(len(st.validators)):
        v = _v(st, i)
        if _active(v, prev) or (v["slashed"] and prev + 1 < v["wd"]):
            out.append(i)
    return out


def _increase(st, i, d):
    st.balances[i] = _check(int(st.balances[i]) + d, "balance")


def _decrease(st, i, d):
    st.balances[i] = max(0, int(st.balances[i]) - d)


def process_epoch_literal(st: SynthState, mask: int = ALL) -> int:
    C = CONSTS[st.preset]
    EBI = C["EFFECTIVE_BALANCE_INCREMENT"]
    try:
        cur, prev = _epochs(st, C)
        n = len(st.validators)
        total = _total_balance(st, [i for i in range(n) if _active(_v(st, i), cur)])   # hoisted get_total_active_balance
        if mask & 1 and cur > 1:
            prev_t = _total_balance(st, _unslashed_participating(st, C, 1, prev, st.previous_epoch_participation))
            cur_t = _total_balance(st, _unslashed_participating(st, C, 1, cur, st.current_epoch_participation))
            weigh_justification_and_finalization(st, C, total, prev_t, cur_t)
        if mask & 2 and cur > 0:
            leak = is_in_inactivity_leak(st, C)
            target = set(_unslashed_participating(st, C, 1, prev, st.previous_epoch_participation))
            for i in _eligible(st, prev):
                s = int(st.inactivity_scores[i])
                if i in target:
                    s -= min(1, s)
                else:
                    s = _check(s + C["INACTIVITY_SCORE_BIAS"], "inactivity score")
                if not leak:
                    s -= min(C["INACTIVITY_SCORE_RECOVERY_RATE"], s)
                st.inactivity_scores[i] = s
        if mask & 4 and cur > 0:
            leak = is_in_inactivity_leak(st, C)
            eligible = _eligible(st, prev)
            brpi = EBI * C["BASE_REWARD_FACTOR"] // integer_squareroot(total)
            deltas = []
            for flag in range(3):   # get_flag_index_deltas
                part = set(_unslashed_participating(st, C, flag, prev, st.previous_epoch_participation))
                part_incr = _total_balance(st, sorted(part)) // EBI
                active_incr = total // EBI
                rw, pn = [0] * n, [0] * n
                for i in eligible:
                    base = _check(_v(st, i)["eb"] // EBI * brpi, "base reward")
                    if i in part:
                        if not leak:
                            num = _check(_check(base * WEIGHTS[flag], "reward") * part_incr, "reward")
                            rw[i] += num // (active_incr * WEIGHT_DENOMINATOR)
                    elif flag != 2:
                        pn[i] += _check(base * WEIGHTS[flag], "penalty") // WEIGHT_DENOMINATOR
                deltas.append((rw, pn))
            target = set(_unslashed_participating(st, C, 1, prev, st.previous_epoch_participation))
            rw, pn = [0] * n, [0] * n   # get_inactivity_penalty_deltas
            for i in eligible:
                if i not in target:
                    num = _check(_v(st, i)["eb"] * int(st.inactivity_scores[i]), "inactivity penalty")
                    pn[i] += num // (C["INACTIVITY_SCORE_BIAS"] * C["INACTIVITY_PENALTY_QUOTIENT_BELLATRIX"])
            deltas.append((rw, pn))
            for rw, pn in deltas:
                for i in range(n):
                    _increase(st, i, rw[i])
                    _decrease(st, i, pn[i])
        if mask & 8:
            active_count = sum(1 for i in range(n) if _active(_v(st, i), cur))
            churn = max(C["MIN_PER_EPOCH_CHURN_LIMIT"], active_count // C["CHURN_LIMIT_QUOTIENT"])
            aee_epoch = cur + 1 + C["MAX_SEED_LOOKAHEAD"]
            V = st.validators
            for i in range(n):
                v = _v(st, i)
                if v["aee"] == FAR_FUTURE_EPOCH and v["eb"] == C["MAX_EFFECTIVE_BALANCE"]:
                    V["activation_eligibility_epoch"][i] = cur + 1
                if _active(v, cur) and v["eb"] <= C["EJECTION_BALANCE"] and v["exit"] == FAR_FUTURE_EPOCH:
                    # initiate_validator_exit: rescans the registry
                    exits = [int(x) for x in V["exit_epoch"] if int(x) != FAR_FUTURE_EPOCH]
                    q = max(exits + [aee_epoch])
                    if sum(1 for x in V["exit_epoch"] if int(x) == q) >= churn:
                        q = _check(q + 1, "exit epoch")
                    V["exit_epoch"][i] = q
                    V["withdrawable_epoch"][i] = _check(q + C["MIN_VALIDATOR_WITHDRAWABILITY_DELAY"], "withdrawable epoch")
            fin = _u64(st.fixed["finalized_checkpoint"])
            queue = [i for i in range(n) if int(V["activation_eligibility_epoch"][i]) <= fin
                     and int(V["activation_epoch"][i]) == FAR_FUTURE_EPOCH]
            queue.sort(key=lambda i: (int(V["activation_eligibility_epoch"][i]), i))
            for i in queue[:min(C["MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT"], churn)]:
                V["activation_epoch"][i] = aee_epoch
        if mask & 16:
            adjusted = min(_check(_check(sum(int(x) for x in st.slashings), "slashings") *
                                  C["PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX"], "slashings"), total)
            for i in range(n):
                v = _v(st, i)
                if v["slashed"] and cur + C["EPOCHS_PER_SLASHINGS_VECTOR"] // 2 == v["wd"]:
                    num = _check(v["eb"] // EBI * adjusted, "slashing penalty")
                    _decrease(st, i, num // total * EBI)
        if mask & 32:
            eth1_data_reset(st, C)
        if mask & 64:
            inc = EBI // C["HYSTERESIS_QUOTIENT"]
            down, up = inc * C["HYSTERESIS_DOWNWARD_MULTIPLIER"], inc * C["HYSTERESIS_UPWARD_MULTIPLIER"]
            for i in range(n):
                b, eb = int(st.balances[i]), _v(st, i)["eb"]
                if _check(b + down, "hysteresis") < eb or _check(eb + up, "hysteresis") < b:
                    st.validators["effective_balance"][i] = min(b - b % EBI, C["MAX_EFFECTIVE_BALANCE"])
        return _tail(st, C, mask)
    except Invalid:
        return INVALID


def _tail(st, C, mask) -> int:
    if mask & 128:
        slashings_reset(st, C)
    if mask & 256:
        randao_mixes_reset(st, C)
    if mask & 512:
        historical_summaries_update(st, C)
    if mask & 1024:
        participation_flag_updates(st, C)
    if mask & 2048:
        return sync_committee_updates(st, C)
    return 0


# ------------------------------------------------------------------------------------------------ numpy form

def _usum(a: np.ndarray) -> int:
    a = a.astype(np.uint64)
    return (int((a >> np.uint64(32)).sum()) << 32) + int((a & np.uint64(0xFFFFFFFF)).sum())


def _mul_ok(a: np.ndarray, b) -> bool:
    """every a * b fits in a uint64 (b scalar or array)"""
    a = a.astype(np.uint64)
    b = np.broadcast_to(np.asarray(b, dtype=np.uint64), a.shape)
    nz = b != 0
    return not np.any(a[nz] > np.uint64(U64) // b[nz])


def process_epoch_numpy(st: SynthState, mask: int = ALL) -> int:
    C = CONSTS[st.preset]
    EBI = C["EFFECTIVE_BALANCE_INCREMENT"]
    u = np.uint64
    try:
        cur, prev = _epochs(st, C)
        V = st.validators
        eb = V["effective_balance"].astype(u)
        slashed = V["slashed"] != 0
        act, ext, wd = V["activation_epoch"].astype(u), V["exit_epoch"].astype(u), V["withdrawable_epoch"].astype(u)
        act_cur = (act <= u(cur)) & (u(cur) < ext)
        act_prev = (act <= u(prev)) & (u(prev) < ext)
        pp = st.previous_epoch_participation
        part = [act_prev & ~slashed & (((pp >> f) & 1) == 1) for f in range(3)]
        floor = lambda x: max(EBI, _check(x, "total balance"))  # noqa: E731
        total = floor(_usum(eb[act_cur]))
        if mask & 1 and cur > 1:
            cp = st.current_epoch_participation
            cur_t = floor(_usum(eb[act_cur & ~slashed & (((cp >> 1) & 1) == 1)]))
            weigh_justification_and_finalization(st, C, total, floor(_usum(eb[part[1]])), cur_t)
        eligible = act_prev | (slashed & (u(prev) + u(1) < wd))
        if mask & 2 and cur > 0:
            leak = is_in_inactivity_leak(st, C)
            s = st.inactivity_scores.astype(u)
            grow = eligible & ~part[1]
            if np.any(s[grow] > u(U64 - C["INACTIVITY_SCORE_BIAS"])):
                raise Invalid("inactivity score")
            s = np.where(eligible & part[1], s - np.minimum(u(1), s), s)
            s = np.where(grow, s + u(C["INACTIVITY_SCORE_BIAS"]), s)
            if not leak:
                s = np.where(eligible, s - np.minimum(u(C["INACTIVITY_SCORE_RECOVERY_RATE"]), s), s)
            st.inactivity_scores = s.astype("<u8")
        if mask & 4 and cur > 0:
            leak = is_in_inactivity_leak(st, C)
            brpi = EBI * C["BASE_REWARD_FACTOR"] // integer_squareroot(total)
            incr = eb // u(EBI)
            if not _mul_ok(incr[eligible], brpi):
                raise Invalid("base reward")
            base = incr * u(brpi)
            b = st.balances.astype(u)
            active_incr = total // EBI
            for f in range(3):
                p_incr = floor(_usum(eb[part[f]])) // EBI
                rw = np.zeros_like(b)
                pn = np.zeros_like(b)
                got = eligible & part[f]
                if not leak:
                    if not _mul_ok(base[got], WEIGHTS[f]) or not _mul_ok(base[got] * u(WEIGHTS[f]), p_incr):
                        raise Invalid("reward")
                    rw[got] = base[got] * u(WEIGHTS[f]) * u(p_incr) // u(active_incr * WEIGHT_DENOMINATOR)
                miss = eligible & ~part[f]
                if f != 2:
                    if not _mul_ok(base[miss], WEIGHTS[f]):
                        raise Invalid("penalty")
                    pn[miss] = base[miss] * u(WEIGHTS[f]) // u(WEIGHT_DENOMINATOR)
                if np.any(b > u(U64) - rw):
                    raise Invalid("balance")
                b = b + rw
                b = np.where(b > pn, b - pn, u(0))
            miss = eligible & ~part[1]
            sc = st.inactivity_scores.astype(u)
            if not _mul_ok(eb[miss], sc[miss]):
                raise Invalid("inactivity penalty")
            pn = np.zeros_like(b)
            pn[miss] = eb[miss] * sc[miss] // u(C["INACTIVITY_SCORE_BIAS"] * C["INACTIVITY_PENALTY_QUOTIENT_BELLATRIX"])
            b = np.where(b > pn, b - pn, u(0))
            st.balances = b.astype("<u8")
        if mask & 8:
            aee = V["activation_eligibility_epoch"].astype(u)
            churn = max(C["MIN_PER_EPOCH_CHURN_LIMIT"], int(act_cur.sum()) // C["CHURN_LIMIT_QUOTIENT"])
            aee_epoch = cur + 1 + C["MAX_SEED_LOOKAHEAD"]
            V["activation_eligibility_epoch"] = np.where((aee == u(FAR_FUTURE_EPOCH)) & (eb == u(C["MAX_EFFECTIVE_BALANCE"])),
                                                         u(cur + 1), aee)
            ej = np.nonzero(act_cur & (eb <= u(C["EJECTION_BALANCE"])) & (ext == u(FAR_FUTURE_EPOCH)))[0]
            if len(ej):
                exits = ext[ext != u(FAR_FUTURE_EPOCH)]
                max_exit = int(exits.max()) if len(exits) else None
                count = int((ext == u(max_exit)).sum()) if max_exit is not None else 0
                for i in ej:
                    q, churn_q = aee_epoch, 0
                    if max_exit is not None and max_exit >= q:
                        q, churn_q = max_exit, count
                    if churn_q >= churn:
                        q, churn_q = _check(q + 1, "exit epoch"), 0
                    V["exit_epoch"][i] = q
                    V["withdrawable_epoch"][i] = _check(q + C["MIN_VALIDATOR_WITHDRAWABILITY_DELAY"], "withdrawable epoch")
                    max_exit, count = q, churn_q + 1
            fin = _u64(st.fixed["finalized_checkpoint"])
            q = np.nonzero((aee <= u(fin)) & (act == u(FAR_FUTURE_EPOCH)))[0]
            order = np.lexsort((q, aee[q]))
            V["activation_epoch"][q[order][:min(C["MAX_PER_EPOCH_ACTIVATION_CHURN_LIMIT"], churn)]] = aee_epoch
        b = st.balances.astype(u)
        if mask & 16:
            wd = V["withdrawable_epoch"].astype(u)   # registry updates may have moved it
            ssum = _check(_usum(st.slashings), "slashings")
            adjusted = min(_check(ssum * C["PROPORTIONAL_SLASHING_MULTIPLIER_BELLATRIX"], "slashings"), total)
            hit = slashed & (wd == u(cur + C["EPOCHS_PER_SLASHINGS_VECTOR"] // 2))
            if not _mul_ok(eb[hit] // u(EBI), adjusted):
                raise Invalid("slashing penalty")
            pn = np.zeros_like(b)
            pn[hit] = eb[hit] // u(EBI) * u(adjusted) // u(total) * u(EBI)
            b = np.where(b > pn, b - pn, u(0))
            st.balances = b.astype("<u8")
        if mask & 32:
            eth1_data_reset(st, C)
        if mask & 64:
            inc = EBI // C["HYSTERESIS_QUOTIENT"]
            down, up = inc * C["HYSTERESIS_DOWNWARD_MULTIPLIER"], inc * C["HYSTERESIS_UPWARD_MULTIPLIER"]
            if np.any(b > u(U64 - down)) or np.any(eb > u(U64 - up)):
                raise Invalid("hysteresis")
            upd = (b + u(down) < eb) | (eb + u(up) < b)
            V["effective_balance"] = np.where(upd, np.minimum(b - b % u(EBI), u(C["MAX_EFFECTIVE_BALANCE"])), eb)
        return _tail(st, C, mask)
    except Invalid:
        return INVALID


# ------------------------------------------------------------------------------------------------ slots

def block_header_root(hdr: bytes) -> bytes:
    leaves = [hdr[0:8].ljust(32, b"\0"), hdr[8:16].ljust(32, b"\0"), hdr[16:48], hdr[48:80], hdr[80:112]]
    return so.merkleize_chunks(leaves, 8)


def process_slots(st: SynthState, slot: int, epoch_fn=process_epoch_numpy) -> int:
    """process_slots (deneb/spec/mod.rs:3150-3240); the state root of each slot from the hashlib oracle."""
    C = CONSTS[st.preset]
    if slot <= _u64(st.fixed["slot"]):
        raise ValueError("TransitionToPreviousSlot")
    while _u64(st.fixed["slot"]) < slot:
        s = _u64(st.fixed["slot"])
        root = state_root(st)
        st.state_roots[s % C["SLOTS_PER_HISTORICAL_ROOT"]] = np.frombuffer(root, np.uint8)
        hdr = st.fixed["latest_block_header"]
        if hdr[48:80] == bytes(32):
            hdr = hdr[:48] + root + hdr[80:]
            st.fixed["latest_block_header"] = hdr
        st.block_roots[s % C["SLOTS_PER_HISTORICAL_ROOT"]] = np.frombuffer(block_header_root(hdr), np.uint8)
        if (s + 1) % C["SLOTS_PER_EPOCH"] == 0:
            rc = epoch_fn(st, ALL)
            if rc:
                return rc
        st.fixed["slot"] = _p64(s + 1)
    return 0


def copy_state(st: SynthState) -> SynthState:
    return copy.deepcopy(st)
