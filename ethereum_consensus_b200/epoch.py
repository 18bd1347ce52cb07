"""deneb `process_epoch` / `process_slots` on a device-resident state (deneb/spec/mod.rs:965-1004, :3150-3240).

The state never leaves HBM: after these calls `DeviceBeaconState.hash_tree_root()` (or the incremental root) is the
post-state root, and `DeviceBeaconState.to_ssz()` returns the post-state when the host needs its copy back.
"""
from __future__ import annotations

from . import _lib
from .crypto import _result

# stage bits, in the order process_epoch runs them
JUSTIFICATION_AND_FINALIZATION = 1 << 0
INACTIVITY_UPDATES = 1 << 1
REWARDS_AND_PENALTIES = 1 << 2
REGISTRY_UPDATES = 1 << 3
SLASHINGS = 1 << 4
ETH1_DATA_RESET = 1 << 5
EFFECTIVE_BALANCE_UPDATES = 1 << 6
SLASHINGS_RESET = 1 << 7
RANDAO_MIXES_RESET = 1 << 8
HISTORICAL_SUMMARIES_UPDATE = 1 << 9
PARTICIPATION_FLAG_UPDATES = 1 << 10
SYNC_COMMITTEE_UPDATES = 1 << 11
ALL = 0xFFF
STAGES = {  # epoch_processing/<handler> names of the consensus spec tests
    "justification_and_finalization": JUSTIFICATION_AND_FINALIZATION, "inactivity_updates": INACTIVITY_UPDATES,
    "rewards_and_penalties": REWARDS_AND_PENALTIES, "registry_updates": REGISTRY_UPDATES, "slashings": SLASHINGS,
    "eth1_data_reset": ETH1_DATA_RESET, "effective_balance_updates": EFFECTIVE_BALANCE_UPDATES,
    "slashings_reset": SLASHINGS_RESET, "randao_mixes_reset": RANDAO_MIXES_RESET,
    "historical_summaries_update": HISTORICAL_SUMMARIES_UPDATE, "participation_flag_updates": PARTICIPATION_FLAG_UPDATES,
    "sync_committee_updates": SYNC_COMMITTEE_UPDATES,
}


class StateTransitionInvalid(ValueError):
    """A uint64 overflow or a failed spec assertion (code 18).  The spec rejects the transition; the handle is failed
    and must be freed and uploaded again."""


class TransitionToPreviousSlot(ValueError):
    """process_slots to a slot that is not after the state's slot."""


def _check(rc: int, where: str) -> None:
    if rc == _lib.STATE_TRANSITION_INVALID:
        raise StateTransitionInvalid(f"{where}: {_lib.load().b200_last_error().decode(errors='replace')}")
    _result(rc, where)   # 1..7: an invalid key in the next sync committee, as crypto.eth_aggregate_public_keys


def process_epoch(dev_state, stages: int = ALL) -> None:
    """Run the process_epoch stages in `stages` (bits above; ALL = process_epoch) on `dev_state` in place."""
    _check(_lib.lib().b200_state_process_epoch_deneb(dev_state._h, int(stages)), "process_epoch")


def process_slots(dev_state, slot: int) -> None:
    """Advance `dev_state` to `slot`, running process_epoch at every epoch boundary."""
    rc = _lib.lib().b200_state_process_slots_deneb(dev_state._h, int(slot))
    if rc == _lib.ERR_BAD_ARG and "TransitionToPreviousSlot" in _lib.load().b200_last_error().decode(errors="replace"):
        raise TransitionToPreviousSlot(f"process_slots: slot {slot} is not after the state's slot")
    _check(rc, "process_slots")
