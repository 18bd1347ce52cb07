"""epoch_processing half of the conformance-vector runner, in the layout of the reference's
spec-tests/runners/epoch_processing.rs: `tests/<config>/deneb/epoch_processing/<handler>/<suite>/<case>/` with
`pre.ssz_snappy` and, when the sub-function succeeds, `post.ssz_snappy` (a missing post means an expected failure).
Each handler applies one process_epoch sub-function.  Test infrastructure only."""
from __future__ import annotations

from pathlib import Path
from typing import Callable, Optional, Tuple

from ethereum_consensus_b200 import state as S
from oracle import epoch_oracle as eo
from tests.spec_vectors import snappy_raw_compress_literal, snappy_raw_decompress

EPOCH_HANDLERS = tuple(eo.STAGES)


def run_epoch_case(config: str, handler: str, case_dir: Path, apply: Callable[[bytes, str, int], Optional[bytes]]) -> Tuple[bool, str]:
    """`apply(pre_ssz, preset, stage_bit)` returns the post-state SSZ, or None when the sub-function fails."""
    if handler not in EPOCH_HANDLERS:
        return True, "skipped handler"
    pre = snappy_raw_decompress((case_dir / "pre.ssz_snappy").read_bytes())
    post_file = case_dir / "post.ssz_snappy"
    want = snappy_raw_decompress(post_file.read_bytes()) if post_file.exists() else None
    got = apply(pre, config, 1 << EPOCH_HANDLERS.index(handler))
    if want is None:
        return got is None, "expected failure"
    return got == want, "post-state"


def oracle_apply(pre: bytes, preset: str, bit: int) -> Optional[bytes]:
    st = eo.from_ssz(pre, preset)
    return None if eo.process_epoch_numpy(st, bit) else S.serialize(st).tobytes()


def synthetic_tree(base: Path, cases) -> Path:
    """One case per (golden scenario, handler) from the oracle: `cases` = [(name, preset, seed, build_state)]."""
    for name, preset, seed, build in cases:
        for bit, handler in enumerate(EPOCH_HANDLERS):
            d = base / "tests" / preset / "deneb" / "epoch_processing" / handler / "pyspec_tests" / name
            d.mkdir(parents=True, exist_ok=True)
            st = build(name, preset, seed)
            (d / "pre.ssz_snappy").write_bytes(snappy_raw_compress_literal(S.serialize(st).tobytes()))
            if eo.process_epoch_numpy(st, 1 << bit) == 0:
                (d / "post.ssz_snappy").write_bytes(snappy_raw_compress_literal(S.serialize(st).tobytes()))
    return base
