"""CPU: the prover's scalar code that the kernels compile — the quotient of csrc/kzg_quotient.cuh (batch inversion and the
in-domain branch) and the signed-digit recoding of csrc/msm.cuh — built for the host and checked against Python ints and
tests/kzg_prover_oracle.py."""
import ctypes
import random
import subprocess
from pathlib import Path

import pytest

from oracle import kzg_oracle as ko
from tests import kzg_prover_oracle as kp

ROOT = Path(__file__).resolve().parent.parent
R = ko.R
EDGE = [0, 1, R - 1, (R - 1) // 2, (R + 1) // 2, 1 << 254, (1 << 254) - 1, 2, R - 2]


@pytest.fixture(scope="module")
def hp(tmp_path_factory):
    src = ROOT / "tests" / "host_math" / "host_kzg_prover.cpp"
    lib = tmp_path_factory.mktemp("host_kzg_prover") / "libhost_kzg_prover.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", str(lib), str(src)], check=True)
    L = ctypes.CDLL(str(lib))
    L.hk_quotient.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p]
    L.hk_inv_root_index.argtypes = [ctypes.c_uint32]
    L.hk_inv_root_index.restype = ctypes.c_uint32
    L.hk_digits.argtypes = [ctypes.c_char_p, ctypes.c_void_p]
    L.hk_digits.restype = ctypes.c_uint32
    return L


def _be(v): return v.to_bytes(32, "big")


def _params(hp):
    out = (ctypes.c_int32 * 4)()
    hp.hk_msm_params(out)
    return list(out)


def _quotient(hp, poly, z, parts):
    blob = b"".join(_be(v) for v in poly)
    y = ko.evaluate_polynomial_in_evaluation_form(poly, z)
    out = ctypes.create_string_buffer(32 * 4096)
    hp.hk_quotient(blob, _be(z), _be(y), parts, out)
    return [int.from_bytes(out.raw[32 * i:32 * i + 32], "big") for i in range(4096)], y


@pytest.mark.parametrize("parts", [1, 256])
def test_quotient_out_of_domain(hp, parts):
    rng = random.Random(3 + parts)
    poly = [rng.randrange(R) for _ in range(4096)]
    for z in [rng.randrange(R), 0, R - 2, (R + 1) // 2, 1 << 254]:
        q, y = _quotient(hp, poly, z, parts)
        assert z not in ko.ROOTS_BRP
        assert q == kp.quotient(poly, z, y), z


@pytest.mark.parametrize("parts", [1, 256])
def test_quotient_in_domain(hp, parts):
    rng = random.Random(5 + parts)
    poly = [rng.randrange(R) for _ in range(4096)]
    for i in (0, 1, 2048, 4095, 1234):   # w_0 = 1, w_2048... : 1 and r - 1 are among them
        z = ko.ROOTS_BRP[i]
        q, y = _quotient(hp, poly, z, parts)
        assert y == poly[i]
        assert q == kp.quotient(poly, z, y), i
    assert ko.ROOTS_BRP[0] == 1 and ko.ROOTS_BRP[1] == R - 1


def test_inverse_root_index(hp):
    for m in list(range(8)) + [2048, 4095, 1234]:
        assert ko.ROOTS_BRP[hp.hk_inv_root_index(m)] * ko.ROOTS_BRP[m] % R == 1, m


def test_signed_digits_recompose(hp):
    c, windows, max_digit, _ = _params(hp)
    rng = random.Random(9)
    vals = EDGE + [rng.randrange(R) for _ in range(500)] + [int("10" * 127, 2), (1 << 255) - 1 - (1 << 200)]
    digits = (ctypes.c_int32 * windows)()
    for s in vals:
        if s >= 1 << 255:
            continue
        carry = hp.hk_digits(_be(s), digits)
        assert carry == 0, hex(s)
        ds = list(digits)
        assert all(-(max_digit - 1) <= d <= max_digit for d in ds), hex(s)
        assert sum(d << (c * w) for w, d in enumerate(ds)) == s, hex(s)
