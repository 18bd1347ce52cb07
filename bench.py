#!/usr/bin/env python
"""bench.py — BASELINE.json's metric on BASELINE.json's configs.

Headline (configs[1]): `fast_aggregate_verify tuples/s`, mainnet preset, T = 4096 attestation tuples x K = 512 public
keys per tuple, strict mode (every key decompressed + validated in every call, as
/root/reference/ethereum-consensus/src/crypto/bls.rs:119-123 does), on 1..N B200 (one process per GPU; tuples shard
with no data-path collective; the per-shard verdict vectors are exchanged with one NCCL all_gather).
Secondary (configs[2]), same JSON line under "ssz": `hash_tree_root(BeaconState) ms`, deneb mainnet, 2**20 validators.

One step = one pass of the hot path over one batch.  `value` = device time (CUDA events on the library's launching
stream, inputs already in HBM); `e2e` = the same batch through the public C-ABI call with pinned HOST buffers,
H2D + kernels + D2H of the verdicts inside the timed region.  `--impl reference` times the CPU restatement
(oracle/, plain C; blst/ssz_rs themselves cannot be built offline — DESIGN.md) on the host cores.
`--dump-outputs DIR` writes the verdict codes and the state root of the last timed step as DIR/<name>.npy.
"""
from __future__ import annotations

import argparse
import atexit
import ctypes as C
import hashlib
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True   # the benchmark leaves the tree as it found it (it may be read-only)

R_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
SEED = 0xB200
# a point of E'(Fp2) outside G2 (iso3(sswu(5+7u)) compressed; produced by oracle/bls_oracle.py, see tests/golden)
SIG_NOT_IN_GROUP = None  # filled from tests/golden/bls_cases.json
# integer-arithmetic SASS instructions per 64-byte pair hash (2 compressions): 2 033 LOP3/SHF/IADD3 + 246 adds / moves the
# compiler places on the FMA pipe (IMAD.IADD, PRMT, ...) — counted by tools/count_sha_sass.py from cuobjdump of the shipped
# k_validator_roots (8 pair hashes of straight-line code per thread; 2 340 instructions in all); the denominator
# b200_measure_int_peak(2) is the same kind of mix, which the compiler also spreads over both pipes (DESIGN.md §4)
SASS_OPS_PER_PAIR_HASH = 2279
ORACLE_BUILD = "gcc -O3"   # set by load_oracles()


# ------------------------------------------------------------------------------------------------ helpers
def load_oracles():
    # the oracles build() compiled under oracle/; when they are missing or older than their sources, this process compiles
    # its own copy into a temporary directory, since the tree may be read-only (and ranks then never share a build)
    lib_dir = ROOT / "oracle"
    if subprocess.run(["make", "-q", "-C", str(lib_dir)], capture_output=True).returncode != 0:
        lib_dir = Path(tempfile.mkdtemp(prefix="b200_oracle_"))
        atexit.register(shutil.rmtree, lib_dir, True)
        subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), f"OUT={lib_dir}/"], check=True)
    # the timed CPU arm gets the mulx / adx build when this host's CPU has both features (same results, ~20 % faster products)
    global ORACLE_BUILD
    try:
        flags = set(next(ln for ln in open("/proc/cpuinfo") if ln.startswith("flags")).split())
    except (OSError, StopIteration):
        flags = set()
    adx = {"adx", "bmi2"} <= flags and (lib_dir / "liboracle_bls_adx.so").exists()
    ORACLE_BUILD = "gcc -O3 -mbmi2 -madx" if adx else "gcc -O3"
    bls = C.CDLL(str(lib_dir / ("liboracle_bls_adx.so" if adx else "liboracle_bls.so")))
    ssz = C.CDLL(str(lib_dir / "liboracle_ssz.so"))
    vp, sz, ci = C.c_void_p, C.c_size_t, C.c_int
    bls.orc_fast_aggregate_verify_batch.argtypes = [vp, vp, vp, vp, sz, vp, ci]
    bls.orc_sign_batch.argtypes = [vp, vp, sz, vp, ci]
    bls.orc_pk_sequence.argtypes = [C.c_char_p, C.c_char_p, sz, vp]
    bls.orc_fast_aggregate_verify.argtypes = [vp, sz, vp, sz, vp]
    bls.orc_fp_mul_count.restype = C.c_uint64
    bls.orc_fp_sqr_count.restype = C.c_uint64
    bls.orc_key_validate.argtypes = [vp]
    ssz.orc_htr_beacon_state_deneb.argtypes = [vp, sz, ci, ci, vp]
    ssz.orc_htr_beacon_state_deneb.restype = ci
    return bls, ssz


def usable_host_threads() -> int:
    """Threads this process may really use: the scheduler affinity mask capped by the cgroup CPU quota (os.cpu_count()
    reports the machine, not the container: round 1 timed "128 threads" on a box that granted ~10 cores' worth)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = Path("/sys/fs/cgroup/cpu.max").read_text().split()
        if quota != "max":
            n = max(1, min(n, int(float(quota) / float(period) + 0.5)))
    except Exception:
        try:
            q = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read_text())
            per = int(Path("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read_text())
            if q > 0:
                n = max(1, min(n, int(q / per + 0.5)))
        except Exception:
            pass
    return n


class ClockSampler:
    """Samples SM clock / power / throttle reasons during the timed region through NVML (pynvml, initialised once).
    Spawning `nvidia-smi` five times a second re-initialises NVML each time and measurably slows the kernels being
    timed (K1 167 -> 186 ms), so the recipe's query is issued through the library instead."""

    def __init__(self, gpu_index: int):
        self.idx, self.rows, self._stop, self._th = gpu_index, [], threading.Event(), None
        self.h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def _run(self):
        nv = self.nv
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.rows.append((sm, pw, rs))
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        if self.h is not None and not os.environ.get("BENCH_NO_SAMPLER"):
            self._th = threading.Thread(target=self._run, daemon=True)
            self._th.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._th is not None:
            self._th.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["NVML unavailable"]}
        nv = self.nv
        sm = sorted(r[0] for r in self.rows)
        bits = 0
        for r in self.rows:
            bits |= r[2]
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        return {"sm_mhz": float(sm[len(sm) // 2]), "sm_min_mhz": float(sm[0]), "sm_max_mhz": float(self.max_sm),
                "power_w_max": max(r[1] for r in self.rows), "samples": len(self.rows),
                "reasons": [k for k, v in names.items() if bits & v]}


from tests import workloads  # noqa: E402
from tests.workloads import make_bls_workload  # noqa: E402  (the workload generator is shared with the parity tests)


def pin(arr):
    import torch
    t = torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
    return t


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir: str, arrays: dict) -> None:
    """--dump-outputs: what the timed paths returned in their last step, as DIR/<name>.npy in float64, so that two builds
    run with the same arguments (hence the same seeded inputs) can be compared output for output.  An array larger than
    its share of DUMP_BYTES is replaced by a fixed, seeded sample of its elements (same positions in every run)."""
    d = Path(out_dir)
    d.mkdir(parents=True, exist_ok=True)
    cap = DUMP_BYTES // 8 // max(1, len(arrays))
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float64).ravel()
        if a.size > cap:
            a = a[np.sort(np.random.default_rng(SEED).choice(a.size, cap, replace=False))]
        np.save(d / f"{name}.npy", a)


# ------------------------------------------------------------------------------------------------ main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--tuples", type=int, default=4096)
    ap.add_argument("--keys", type=int, default=512)
    ap.add_argument("--validators", type=int, default=1 << 20)
    ap.add_argument("--skip-ssz", action="store_true")
    ap.add_argument("--skip-strong", action="store_true", help="skip the configs[4] strong-scaling batch")
    ap.add_argument("--skip-single", action="store_true", help="skip the single-call latency probe")
    ap.add_argument("--skip-rlc", action="store_true", help="skip the RLC whole-batch check")
    ap.add_argument("--skip-block", action="store_true", help="skip the configs[3] block signature set")
    ap.add_argument("--strong-tuples", type=int, default=2048)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write each timed path's last outputs to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    # Libraries (NCCL's version banner, make, ...) may write to fd 1; the contract is ONE JSON line on stdout from rank 0.
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    host_threads = usable_host_threads()
    T, K = args.tuples, args.keys
    workload = f"mainnet preset: batch {T} Attestation fast_aggregate_verify tuples, K={K} pubkeys/tuple, strict per-key validation"
    base = {"metric": "fast_aggregate_verify tuples/s", "unit": "tuples/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 limbs (381-bit Fp), u32 SHA-256 words",
            "data": "synthetic",
            "config": {"workload": workload, "tuples_per_gpu": T, "keys_per_tuple": K, "registry": 1 << 20, "mode": "strict",
                       "adversarial_fraction": 0.03, "l2": "256 MiB memset between timed steps (flush)", "parallelism": f"tuples sharded x{world}"}}

    orc_bls, orc_ssz = load_oracles()

    # ---------------------------------------------------------------- reference arm: CPU restatement on host cores
    if args.impl == "reference":
        if rank != 0:
            return
        sample = min(T, 8 * host_threads)
        w = make_bls_workload(orc_bls, sample, K, 0, threads=host_threads)
        out = np.empty(sample, dtype=np.int32)
        times = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            orc_bls.orc_fast_aggregate_verify_batch(w["pks"].ctypes.data, w["off"].ctypes.data, w["msgs"].ctypes.data, w["sigs"].ctypes.data,
                                                    sample, out.ctypes.data, host_threads)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
        assert out.tolist() == w["expect"].tolist(), "CPU restatement disagrees with the constructed verdicts"
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {"fast_aggregate_verify_codes": out})
        ms = 1e3 * sum(times) / len(times)
        v = sample / (ms / 1e3)
        line = dict(base)
        line.update({"impl": "reference", "value": v, "ms_per_step": ms, "gpu_launches": 0,
                     "cpu_baseline": {"value": v, "unit": "tuples/s", "cores": host_threads, "kind": "port",
                                      "sample": f"{sample} of the {T} tuples per step, all host threads (plain-C restatement built with {ORACLE_BUILD}, not blst)"},
                     "e2e": {"value": v, "unit": "tuples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        emit(line)
        return

    # ---------------------------------------------------------------- our arm
    import torch
    import torch.distributed as dist
    from ethereum_consensus_b200 import _lib, crypto, parallel, ssz, state as S

    torch.cuda.set_device(local_rank)
    if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
        os.environ["NCCL_DEBUG"] = "WARN"  # keep NCCL's version banner off stdout: rank 0 prints exactly one JSON line
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    _lib.init(local_rank)
    lib = _lib.load()
    # the library's own communicator: every data-path exchange below is a collective issued by the C library on its
    # engine stream (comm.cu); torch.distributed only carries the 128-byte NCCL id and the timing barriers
    parallel.comm_init(rank, world)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def flush_l2():
        if os.environ.get("BENCH_NO_FLUSH"):   # diagnostics only; the default run flushes
            return
        flush_buf.zero_()
        torch.cuda.synchronize()

    w = make_bls_workload(orc_bls, T, K, rank, threads=host_threads)
    pks, off, msgs, sigs = pin(w["pks"]), w["off"], pin(w["msgs"]), pin(w["sigs"])

    def step():
        codes = crypto.fast_aggregate_verify_batch(pks, off, msgs, sigs)
        if world > 1:  # the path's one exchange step: every rank learns every shard's verdicts (ncclAllGather in the library)
            everyone = parallel.comm_all_gather_codes(codes)
            assert len(everyone) == world * T
        return codes

    for _ in range(args.warmup):
        codes = step()
    assert codes.tolist() == w["expect"].tolist(), "GPU verdicts differ from the constructed expectation"

    launches0, coll0 = lib.b200_launch_count(), lib.b200_collective_count()
    dev_ms, dom_ms, wall = [], [], []
    with ClockSampler(local_rank) as clk:
        barrier()
        t_all0 = time.perf_counter()
        for _ in range(args.steps):
            flush_l2()
            barrier()
            t0 = time.perf_counter()
            codes = step()
            barrier()
            wall.append(time.perf_counter() - t0)
            dev_ms.append(crypto.last_kernel_ms())
            dom_ms.append(crypto.last_dominant_kernel_ms())
        t_all = time.perf_counter() - t_all0
    launches = lib.b200_launch_count() - launches0
    collectives = lib.b200_collective_count() - coll0
    assert codes.tolist() == w["expect"].tolist()

    ms_dev = max_over_ranks(sum(dev_ms) / len(dev_ms))
    ms_e2e = max_over_ranks(1e3 * sum(wall) / len(wall))
    value = world * T / (ms_dev / 1e3)
    e2e_value = world * T / (ms_e2e / 1e3)
    h2d = int(w["pks"].nbytes + w["msgs"].nbytes + w["sigs"].nbytes + w["off"].nbytes)

    # registry mode (validated keys resident in HBM) — reported separately, never as the headline
    reg_ms = None
    try:
        reg = crypto.Registry(pin(w["registry"]))
        reg_load_ms = crypto.last_kernel_ms()
        for _ in range(2):
            rc = reg.verify_batch(w["idx"], off, msgs, sigs)
        reg_ms = crypto.last_kernel_ms()
        # tuples whose bytes were edited (infinity key / cancelling keys) differ by construction in registry mode
        same = (w["kind"] != 4) & (w["kind"] != 5)
        assert (rc[same] == w["expect"][same]).all()
    except Exception as e:  # noqa: BLE001
        reg_ms, reg_load_ms = None, None
        print(f"[bench] registry mode skipped: {e}", file=sys.stderr)

    # ---- BASELINE configs[4]: ONE epoch-scale batch (32 slots x 64 committees = 2048 tuples, K = 512) sharded over the
    # N GPUs — STRONG scaling: total work fixed, every rank holds the same batch, verifies its contiguous block and the
    # library all-gathers the verdicts (b200_fast_aggregate_verify_batch_sharded).  Measured at every N, N = 1 included.
    strong = None
    if not args.skip_strong:
        TS = args.strong_tuples
        ws = make_bls_workload(orc_bls, TS, K, 10_000, threads=host_threads)   # the same batch on every rank
        spk, soff, smsg, ssig = pin(ws["pks"]), ws["off"], pin(ws["msgs"]), pin(ws["sigs"])
        for _ in range(2):
            sc = parallel.sharded_verify_batch(spk, soff, smsg, ssig)
        assert sc.tolist() == ws["expect"].tolist(), "sharded verdicts differ from the constructed expectation"
        s_wall, s_dev = [], []
        for _ in range(args.steps):
            flush_l2()
            barrier()
            t0 = time.perf_counter()
            sc = parallel.sharded_verify_batch(spk, soff, smsg, ssig)
            barrier()
            s_wall.append(time.perf_counter() - t0)
            s_dev.append(crypto.last_kernel_ms())
        assert sc.tolist() == ws["expect"].tolist()
        s_ms = max_over_ranks(1e3 * sum(s_wall) / len(s_wall))
        s_dev_ms = max_over_ranks(sum(s_dev) / len(s_dev))
        lo_t, hi_t = parallel.tuple_shard(TS, world, rank)
        strong = {"workload": f"BASELINE configs[4]: one batch of {TS} tuples (32 slots x 64 committees), K={K}, strict, sharded over {world} GPU(s)",
                  "scaling": "strong", "tuples": TS, "tuples_per_s_e2e": TS / (s_ms / 1e3), "ms_per_batch_e2e": s_ms,
                  "ms_per_batch_device": s_dev_ms, "tuples_per_s_device": TS / (s_dev_ms / 1e3),
                  "h2d_bytes_per_rank": int((hi_t - lo_t) * (48 * K + 128)), "exchange": "ncclAllGather of int32 verdicts inside the library",
                  "checked": "all verdicts equal the constructed expectation on every rank"}

    # ---- RLC whole-batch check (north_star's fused multi-pairing): the all-valid part of the workload, one boolean
    rlc = None
    if rank == 0 and not args.skip_rlc:
        okm = np.nonzero(w["kind"] == 0)[0]
        rp = pin(w["pks"].reshape(T, K * 48)[okm].reshape(-1).copy())
        ro = (np.arange(len(okm) + 1, dtype=np.uint64) * K).astype(np.uint32)
        rm = pin(w["msgs"].reshape(T, 32)[okm].reshape(-1).copy())
        rs = pin(w["sigs"].reshape(T, 96)[okm].reshape(-1).copy())
        seed = hashlib.sha256(b"b200/bench/rlc").digest()
        assert crypto.fast_aggregate_verify_batch_all(rp, ro, rm, rs, seed=seed) is True
        assert crypto.fast_aggregate_verify_batch_all(pks, off, msgs, sigs, seed=seed) is False   # the adversarial mix
        r_dev, r_dom = [], []
        for _ in range(3):
            flush_l2()
            assert crypto.fast_aggregate_verify_batch_all(rp, ro, rm, rs, seed=seed) is True
            r_dev.append(crypto.last_kernel_ms()); r_dom.append(crypto.last_dominant_kernel_ms())
        p_dev = []
        for _ in range(3):
            flush_l2()
            assert (crypto.fast_aggregate_verify_batch(rp, ro, rm, rs) == 0).all()
            p_dev.append(crypto.last_kernel_ms())
        rlc = {"tuples": int(len(okm)), "what": "all-valid subset of the workload; one boolean for the batch (T Miller loops + 1 final exponentiation)",
               "ms_per_batch_device": sum(r_dev) / 3, "ms_per_key_kernel": sum(r_dom) / 3,
               "ms_per_tuple_path_same_batch_device": sum(p_dev) / 3,
               "tuples_per_s_device": len(okm) / (sum(r_dev) / 3 / 1e3)}

    # ---- single-call drop-in latency (the per-call path a straight `crypto::fast_aggregate_verify` replacement takes)
    single = None
    if rank == 0 and not args.skip_single:
        single = {}
        for kk in (1, 512):
            kk = min(kk, K)
            pk_list = [bytes(w["pks"][48 * i: 48 * i + 48]) for i in range(int(w["off"][0]), int(w["off"][0]) + kk)]
            # a valid single tuple: reuse tuple 0's keys only when kk == K, else verify a fresh K=kk tuple from the oracle
            if kk == K and w["kind"][0] == 0:
                m, sg, want = bytes(w["msgs"][:32]), bytes(w["sigs"][:96]), 0
            else:
                m, sg = bytes(w["msgs"][:32]), bytes(w["sigs"][:96])
                arr = np.frombuffer(b"".join(pk_list), dtype=np.uint8)
                want = int(orc_bls.orc_fast_aggregate_verify(arr.ctypes.data, kk, np.frombuffer(m, dtype=np.uint8).ctypes.data, 32,
                                                             np.frombuffer(sg, dtype=np.uint8).ctypes.data))
            ts = []
            for i in range(7):
                t0 = time.perf_counter()
                try:
                    crypto.fast_aggregate_verify(pk_list, m, sg)
                    got = 0
                except crypto.InvalidSignature:
                    got = 5
                except crypto.BLSTError as ex:
                    got = ex.code
                if i >= 2:
                    ts.append((time.perf_counter() - t0) * 1e3)
                assert got == want, (kk, got, want)
            single[f"K={kk}"] = {"ms_per_call": sorted(ts)[len(ts) // 2], "code": want}

    # ---- BASELINE configs[3]: the deneb process_block signature set at spec shape (215 checks), through the host-side
    # collector, host buffers in, code vector out; strict (every key decompressed + validated) and registry mode
    blockset = None
    if rank == 0 and not args.skip_block:
        breg, rows = workloads.make_deneb_block_plan(orc_bls, threads=host_threads)
        sset = workloads.collect_block_signature_set(breg, rows)
        want = [r["expect"] for r in rows]
        reg_b = crypto.Registry(breg.reshape(-1))
        blockset = {"checks": len(rows), "keys_named": int(sum(len(e.pubkeys) for e in sset.entries)),
                    "what": "1 proposer + 1 randao + 32 slashing headers + 4 x K=2048 + 128 x K=512 + 16 deposits + 16 exits + 16 changes "
                            "+ sync aggregate; wall time of SignatureSet.verify() (Python packing + H2D + kernels + D2H)"}
        for mode, kw in (("strict", {}), ("registry", {"registry": reg_b})):
            ts, dev = [], []
            for i in range(7):
                flush_l2()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                got = sset.verify(**kw)
                dt = (time.perf_counter() - t0) * 1e3
                assert got.tolist() == want, f"block signature set ({mode}) differs from the constructed expectation"
                if i >= 2:
                    ts.append(dt); dev.append(crypto.last_kernel_ms())
            blockset[f"ms_per_block_{mode}"] = sorted(ts)[len(ts) // 2]
            blockset[f"ms_last_call_device_{mode}"] = sorted(dev)[len(dev) // 2]
        assert sset.first_failure(got) is None

    line = dict(base)
    peaks = {}
    if rank == 0:
        # ---- CPU baseline: bounded sample of the same workload on the host cores (all threads) + parity on that sample
        sample = min(T, 8 * host_threads)
        out = np.empty(sample, dtype=np.int32)
        t0 = time.perf_counter()
        orc_bls.orc_fast_aggregate_verify_batch(w["pks"].ctypes.data, w["off"].ctypes.data, w["msgs"].ctypes.data, w["sigs"].ctypes.data,
                                                sample, out.ctypes.data, host_threads)
        cpu_dt = time.perf_counter() - t0
        assert out.tolist() == codes[:sample].tolist(), "GPU vs CPU-oracle verdict mismatch on the baseline sample"
        bad = np.nonzero(w["kind"] != 0)[0][:16]  # every adversarial kind, checked against the oracle as well
        for t in bad:
            got = orc_bls.orc_fast_aggregate_verify(w["pks"].ctypes.data + int(w["off"][t]) * 48, K, w["msgs"].ctypes.data + 32 * int(t), 32,
                                                    w["sigs"].ctypes.data + 96 * int(t))
            assert got == int(codes[t]), (int(t), got, int(codes[t]))
        t0 = time.perf_counter()
        orc_bls.orc_fp_mul_count_reset()
        orc_bls.orc_fast_aggregate_verify(w["pks"].ctypes.data, K, w["msgs"].ctypes.data, 32, w["sigs"].ctypes.data)
        cpu_1t = time.perf_counter() - t0
        fp_mul_per_tuple = int(orc_bls.orc_fp_mul_count())
        fp_sqr_per_tuple = int(orc_bls.orc_fp_sqr_count())
        orc_bls.orc_fp_mul_count_reset()
        orc_bls.orc_key_validate(w["pks"].ctypes.data)
        fp_mul_per_key = int(orc_bls.orc_fp_mul_count())   # one key_validate: what the dominant kernel does per thread
        fp_sqr_per_key = int(orc_bls.orc_fp_sqr_count())   # ... of which squarings (222 wide MADs each instead of 288)
        mads_per_key = (fp_mul_per_key - fp_sqr_per_key) * 288 + fp_sqr_per_key * 222

        # integer-pipe denominators (DESIGN.md §4): IMAD.WIDE.U32 issues at one warp instruction per 4 cycles per SM
        # sub-partition = 32 lane-MADs / clk / SM (B300_MICROARCH "rt_SMSP"); the microbenchmarks are the measured
        # cross-check (kind 7: multiplicand from another chain; kind 0: round 1's self-dependent variant)
        clocks = clk.summary()
        sm_mhz = clocks.get("sm_mhz") or 1965.0
        n_sm = torch.cuda.get_device_properties(local_rank).multi_processor_count
        imad_issue_peak = n_sm * 32 * sm_mhz * 1e6 / 1e9           # G wide-MAD/s at the clock seen during the run
        imad_meas = {"self_dependent": crypto.measure_int_peak(0), "cross_chain": crypto.measure_int_peak(7),
                     "cross_chain_immediate": crypto.measure_int_peak(8)}
        alu_peak = crypto.measure_int_peak(2)
        try:
            peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        dom = sum(dom_ms) / len(dom_ms)
        alg_bytes = T * (48 * K + 128)
        k1_mads = T * K * mads_per_key / (dom / 1e3) / 1e9   # algorithmic G MAD/s of the dominant kernel, per launch
        imad_peak = max(imad_issue_peak, max(imad_meas.values()))
        ncu_traffic = None
        try:   # dram__bytes_read.sum + dram__bytes_write.sum of this kernel from the committed ncu capture of THIS build
            ncu_traffic = json.loads((ROOT / "profiles" / "r2_k1_traffic.json").read_text()).get(f"T{T}_K{K}")
        except Exception:
            pass
        line.update({
            "value": value, "ms_per_step": ms_dev, "gpu_launches": int(launches), "nccl_collectives_in_library": int(collectives),
            "e2e": {"value": e2e_value, "unit": "tuples/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4 * T},
            "clocks": clocks,
            # the LIMITING roofline of this path is the FMA-heavy integer pipe (DESIGN.md §4), not HBM: per launch of the
            # dominant kernel, algorithmic 32x32->64 multiply-adds (CPU oracle's instrumented product count for one
            # key_validate x 288) / that kernel's CUDA-event duration, against the IMAD.WIDE issue rate
            "roofline": {"bound": "imad", "kernel": {"7": "k_g1_validate_r168", "0": "k_g1_validate_main", "6": "k_g1_validate_r128"}.get(os.environ.get("B200_G1_VARIANT", "7"), "k_g1_validate"), "achieved": k1_mads, "peak": imad_peak,
                         "unit": "G multiply-adds/s", "frac": k1_mads / imad_peak,
                         "peak_source": "IMAD.WIDE.U32 issue rate: 32 lane-MADs/clk/SM x SMs x SM clock sampled during the run "
                                        "(the larger of that and the on-device microbenchmarks)",
                         "peak_measured_microbench": imad_meas, "peak_issue_rate_model": imad_issue_peak,
                         "fp_products_per_key": fp_mul_per_key, "of_which_squarings": fp_sqr_per_key,
                         "mads_per_product": 288, "mads_per_squaring": 222, "mads_per_key": mads_per_key,
                         "traffic": ncu_traffic, "algorithmic_bytes": T * K * (48 + 104),
                         "kernel_ms": dom, "share_of_step": dom / ms_dev},
            "hbm_roofline": {"bound": "hbm", "achieved": alg_bytes / (dom / 1e3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                             "frac": alg_bytes / (dom / 1e3) / 1e9 / hbm_peak,
                             "peak_source": "measured (MEASURED_PEAKS.json)" if peaks else "fallback",
                             "note": "not the binding limit: 48 B in + 104 B out per key against ~440 k multiply-adds"},
            "int_roofline": {"unit": "G 32x32 multiply-adds/s", "fp_mul_per_tuple_cpu_oracle_count": fp_mul_per_tuple,
                             "squarings_per_tuple": fp_sqr_per_tuple,
                             "achieved": value * ((fp_mul_per_tuple - fp_sqr_per_tuple) * 288 + fp_sqr_per_tuple * 222) / 1e9 / world, "peak": imad_peak,
                             "frac": value * ((fp_mul_per_tuple - fp_sqr_per_tuple) * 288 + fp_sqr_per_tuple * 222) / 1e9 / world / imad_peak,
                             "note": "whole step (all kernels + copies): algorithmic Fp products per tuple (288 MADs, squarings 222) / device time per step",
                             "alu_lop3_shf_iadd3_peak_gops": alu_peak},
            "cpu_baseline": {"value": sample / cpu_dt, "unit": "tuples/s", "cores": host_threads, "kind": "port",
                             "sample": f"first {sample} of the {T} tuples, {host_threads} host threads (affinity/cgroup-limited; machine has "
                                       f"{os.cpu_count()}); single-thread: {1.0 / cpu_1t:.2f} tuples/s, parallel speed-up "
                                       f"{(sample / cpu_dt) * cpu_1t:.1f}x (plain-C restatement of the reference semantics with a dedicated "
                                       f"squaring, built with {ORACLE_BUILD}; no hand assembly: blst is ~1.5x faster per core)"},
            "registry_mode": {"ms_per_step": reg_ms, "tuples_per_s": (T / (reg_ms / 1e3)) if reg_ms else None, "registry_load_ms": reg_load_ms},
            "single_call_latency": single, "rlc_batch_all": rlc, "block_signature_set": blockset,
            "wall_s_timed_region": t_all,
        })
    if strong is not None:
        line["epoch_batch_strong"] = strong
    outputs = {"fast_aggregate_verify_codes": codes}
    if strong is not None:
        outputs["epoch_batch_codes"] = sc

    # ---------------------------------------------------------------- secondary: hash_tree_root(BeaconState)
    if not args.skip_ssz:
        st = S.synth_state(args.validators, "mainnet")
        ssz_bytes = S.serialize(st)
        host = pin(ssz_bytes)
        golden = json.loads((ROOT / "tests" / "golden" / "ssz_roots.json").read_text()).get("mainnet:1048576:default")
        incremental = None
        shuffle_stats = None
        resident_sharded = None
        if world == 1:
            dev = ssz.DeviceBeaconState(host, "mainnet")
            for _ in range(3):
                root = dev.hash_tree_root()
            ks = []
            for _ in range(args.steps):
                flush_l2()
                root = dev.hash_tree_root()
                ks.append(float(lib.b200_last_kernel_ms()))
            # incremental re-hash after one block's worth of writes (SURVEY.md §8f-2): one slot's attesters get a
            # participation flag (N/32 scattered bytes), the sync committee + proposer a new balance, a few Validator
            # records change, plus slot / block_roots / state_roots / randao_mixes entries.  Checked against a full
            # from-scratch hash of the identically patched serialization.
            N = args.validators
            lay = S.layout(st)
            rng = np.random.default_rng(7)
            inc_ms, inc_dev = [], []
            patched = ssz_bytes.copy()
            for it in range(args.steps + 1):
                att = np.unique(rng.choice(N, max(1, N // 32))).astype(np.uint64)
                flags = rng.integers(1, 8, len(att)).astype(np.uint8)
                bal_i = np.unique(rng.choice(N, min(N, 513))).astype(np.uint64)
                bal_v = rng.integers(31 * 10**9, 33 * 10**9, len(bal_i)).astype("<u8")
                val_i = np.unique(rng.choice(N, min(N, 4))).astype(np.uint64)
                vo = lay["validators"][0]
                recs = np.stack([patched[vo + 121 * int(i): vo + 121 * int(i) + 121] for i in val_i]).copy()
                recs[:, 80:88] = np.frombuffer((32 * 10**9 - it - 1).to_bytes(8, "little"), dtype=np.uint8)
                small = [(lay["slot"][0], int(9_000_000 + it).to_bytes(8, "little"))]
                for name in ("block_roots", "state_roots", "randao_mixes"):
                    small.append((lay[name][0] + 32 * (it % 64), rng.integers(0, 256, 32, dtype=np.uint8).tobytes()))
                flush_l2()
                t0 = time.perf_counter()
                dev.update_elements("current_epoch_participation", att, flags)
                dev.update_elements("balances", bal_i, bal_v)
                dev.update_elements("validators", val_i, recs)
                for off_b, data in small:
                    dev.update_bytes(off_b, data)
                inc_root = dev.hash_tree_root_incremental()
                if it:
                    inc_ms.append((time.perf_counter() - t0) * 1e3)
                    inc_dev.append(float(lib.b200_last_kernel_ms()))
                po = lay["current_epoch_participation"][0]
                patched[po + att.astype(np.int64)] = flags
                bo = lay["balances"][0]
                patched[bo: bo + 8 * N].view("<u8")[bal_i.astype(np.int64)] = bal_v
                for i, r in zip(val_i, recs):
                    patched[vo + 121 * int(i): vo + 121 * int(i) + 121] = r
                for off_b, data in small:
                    patched[off_b: off_b + len(data)] = np.frombuffer(data, dtype=np.uint8)
            assert inc_root == ssz.hash_tree_root_beacon_state(patched, "mainnet"), "incremental root differs from the full re-hash"
            incremental = {"ms_per_block_e2e": sum(inc_ms) / len(inc_ms), "ms_device_root_only": sum(inc_dev) / len(inc_dev),
                           "writes_per_block": {"participation_flags": int(max(1, N // 32)), "balances": int(min(N, 513)), "validators": int(min(N, 4)),
                                                "small_fields": 4},
                           "checked_against": "full from-scratch GPU hash of the patched serialization"}
            # committee shuffling on the resident state (SURVEY.md §8f-3): active-index compaction + 90-round shuffle of
            # the whole registry, the per-epoch step before the BLS hot path; checked against the numpy oracle
            from ethereum_consensus_b200 import shuffling as shf
            from oracle import shuffle_oracle as sho
            sh_seed = hashlib.sha256(b"b200/bench/shuffle").digest()
            sh_epoch = 1 << 18
            sh_ms = []
            for _ in range(4):
                flush_l2()
                t0 = time.perf_counter()
                shuffled = shf.state_shuffled_active_indices(dev, sh_epoch, sh_seed, 90)
                sh_ms.append(((time.perf_counter() - t0) * 1e3, float(lib.b200_last_kernel_ms())))
            vo, vl = lay["validators"]
            t0 = time.perf_counter()
            act = np.array(sho.get_active_validator_indices(bytes(ssz_bytes[vo: vo + vl]), sh_epoch), dtype=np.uint64)
            want_sh = sho.shuffled_indices_numpy(act, sh_seed, 90)
            sh_cpu = (time.perf_counter() - t0) * 1e3
            assert np.array_equal(shuffled, want_sh), "shuffled active indices differ from the oracle"
            shuffle_stats = {"validators": N, "active": int(len(act)), "rounds": 90,
                             "ms_device": min(m[1] for m in sh_ms[1:]), "ms_e2e_incl_d2h_of_indices": min(m[0] for m in sh_ms[1:]),
                             "cpu_oracle_ms_numpy_1_thread": sh_cpu, "checked_against": "oracle/shuffle_oracle.py (numpy per-index map)"}
            dev.close()
            es = []
            for i in range(args.steps + 2):
                flush_l2()
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                root2 = ssz.hash_tree_root_beacon_state(host, "mainnet")
                dt = time.perf_counter() - t0
                if i >= 2:
                    es.append(dt * 1e3)
            assert root == root2
            # the same state through the sharded entry point at world = 1 (exercises the exchange plumbing on one GPU)
            assert parallel.sharded_state_root(host, "mainnet") == root
        else:
            ks, es = [], []
            for i in range(args.steps + 3):
                flush_l2()
                barrier()
                t0 = time.perf_counter()
                root = parallel.sharded_state_root(host, "mainnet")   # ONE C-ABI call per rank, NCCL inside the library
                barrier()
                dt_ms = (time.perf_counter() - t0) * 1e3
                if i >= 3:
                    es.append(max_over_ranks(dt_ms))
                    ks.append(max_over_ranks(float(lib.b200_last_kernel_ms())))
            # the same state resident across the ranks: kernels + one ncclAllGather, no PCIe traffic
            sdev = ssz.DeviceBeaconState(host, "mainnet", sharded=True)
            rs = []
            for i in range(args.steps + 3):
                flush_l2()
                barrier()
                t0 = time.perf_counter()
                root_r = sdev.hash_tree_root()
                barrier()
                if i >= 3:
                    rs.append((max_over_ranks((time.perf_counter() - t0) * 1e3), max_over_ranks(float(lib.b200_last_kernel_ms()))))
            assert root_r == root
            sdev.close()
            resident_sharded = {"ms_wall_max_over_ranks": sum(r[0] for r in rs) / len(rs), "ms_device_max_over_ranks": sum(r[1] for r in rs) / len(rs)}
        if args.validators == 1 << 20 and golden:
            assert root.hex() == golden, "hash_tree_root(BeaconState) differs from the hashlib golden root"
        outputs["beacon_state_root"] = np.frombuffer(root, dtype=np.uint8)
        if rank == 0:
            out32 = C.create_string_buffer(32)
            t0 = time.perf_counter()
            orc_ssz.orc_htr_beacon_state_deneb(ssz_bytes.ctypes.data, len(ssz_bytes), 0, 1, out32)
            cpu1 = (time.perf_counter() - t0) * 1e3
            t0 = time.perf_counter()
            orc_ssz.orc_htr_beacon_state_deneb(ssz_bytes.ctypes.data, len(ssz_bytes), 0, host_threads, out32)
            cpun = (time.perf_counter() - t0) * 1e3
            assert out32.raw == root
            n_hash = 10_117_927 if args.validators == 1 << 20 else None
            k_ms = (sum(ks) / len(ks)) if ks else None
            alu_peak_ssz = crypto.measure_int_peak(2)
            hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
            # SHA-256 is ALU-pipe bound: SASS_OPS_PER_PAIR_HASH LOP3/SHF/IADD3-class instructions per 64-byte pair hash
            # (two compressions; counted from cuobjdump of k_merkle_stage, DESIGN.md §4) against the measured issue rate
            # of that instruction mix on this GPU (b200_measure_int_peak(2))
            ops = n_hash * SASS_OPS_PER_PAIR_HASH if n_hash else None
            single_gpu = world == 1
            line["ssz"] = {"metric": "hash_tree_root(BeaconState) ms", "validators": args.validators, "root": root.hex(),
                           "value_ms_device_resident": k_ms if single_gpu else None,
                           "value_ms_device_sharded": None if single_gpu else k_ms,
                           "resident_sharded": resident_sharded,
                           "e2e_ms_from_pinned_host": sum(es) / len(es), "h2d_bytes": int(len(ssz_bytes)),
                           "scaling": "strong" if world > 1 else None,
                           "exchange": None if single_gpu else "one ncclAllGather of 5 x 32 B per rank inside b200_htr_beacon_state_deneb_sharded",
                           "incremental": incremental, "shuffling": shuffle_stats if single_gpu else None,
                           "roofline": {"bound": "alu", "unit": "G ALU instructions/s (LOP3/SHF/IADD3 mix)",
                                        "achieved": (ops / (k_ms / 1e3) / 1e9) if (single_gpu and k_ms and ops) else None,
                                        "peak": alu_peak_ssz,
                                        "frac": (ops / (k_ms / 1e3) / 1e9 / alu_peak_ssz) if (single_gpu and k_ms and ops) else None,
                                        "sass_ops_per_pair_hash": SASS_OPS_PER_PAIR_HASH, "pair_hashes": n_hash,
                                        "sha256_compressions_per_s": (2 * n_hash / (k_ms / 1e3)) if (single_gpu and k_ms and n_hash) else None,
                                        "peak_source": "measured on this GPU (b200_measure_int_peak(2))"},
                           "hbm_roofline": {"bound": "hbm", "achieved": (n_hash * 96 / (k_ms / 1e3) / 1e9) if (single_gpu and k_ms and n_hash) else None,
                                            "peak": hbm_peak, "unit": "GB/s",
                                            "frac": (n_hash * 96 / (k_ms / 1e3) / 1e9 / hbm_peak) if (single_gpu and k_ms and n_hash) else None,
                                            "note": "algorithmic bytes = 10 117 927 pair-hashes x 96 B (SURVEY.md §8d); not the binding limit"},
                           "cpu_baseline": {"ms_1_thread": cpu1, f"ms_{host_threads}_threads": cpun, "kind": "port",
                                            "note": "plain-C restatement with SHA-NI when the host has it (not ssz_rs)"}}
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        emit(line)
    parallel.comm_destroy()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
