"""CPU: the KZG scalar-field arithmetic (csrc/fr.cuh) and the blob evaluation (csrc/kzg_eval.cuh) that the kernels compile,
built for the host and checked against Python ints and the oracle's evaluate_polynomial_in_evaluation_form."""
import ctypes
import random
import subprocess
from pathlib import Path

import pytest

from oracle import kzg_oracle as ko

ROOT = Path(__file__).resolve().parent.parent
R = ko.R
EDGE = [0, 1, 2, R - 1, R - 2, (R - 1) // 2, (R + 1) // 2, 1 << 254, (1 << 254) + 1, (1 << 128) - 1, 1 << 32, (1 << 32) - 1]


@pytest.fixture(scope="module")
def hk(tmp_path_factory):
    src = ROOT / "tests" / "host_math" / "host_kzg.cpp"
    lib = tmp_path_factory.mktemp("host_kzg") / "libhost_kzg.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-fvisibility=hidden", "-o", str(lib), str(src)], check=True)
    L = ctypes.CDLL(str(lib))
    L.hk_fr_op.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_char_p, ctypes.c_char_p]
    L.hk_fr_from_be32.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    L.hk_fr_reduce.argtypes = [ctypes.c_char_p, ctypes.c_char_p]
    L.hk_root_brp.argtypes = [ctypes.c_uint32, ctypes.c_char_p]
    L.hk_eval.argtypes = [ctypes.c_char_p, ctypes.c_char_p, ctypes.c_uint32, ctypes.c_char_p]
    return L


def _be(v): return v.to_bytes(32, "big")


def _op(hk, op, a, b=0):
    out = ctypes.create_string_buffer(32)
    hk.hk_fr_op(op, _be(a), _be(b), out)
    return int.from_bytes(out.raw, "big")


def test_fr_ops_edge_and_random(hk):
    rng = random.Random(1)
    vals = EDGE + [rng.randrange(R) for _ in range(200)]
    pairs = [(a, b) for a in EDGE for b in EDGE] + [(rng.choice(vals), rng.choice(vals)) for _ in range(2000)]
    for a, b in pairs:
        assert _op(hk, 0, a, b) == a * b % R, (a, b)
        assert _op(hk, 3, a, b) == (a + b) % R, (a, b)
        assert _op(hk, 4, a, b) == (a - b) % R, (a, b)
    for a in vals:
        assert _op(hk, 1, a) == a * a % R, a
        assert _op(hk, 5, a) == -a % R, a
        assert _op(hk, 2, a) == (pow(a, -1, R) if a else 0), a


def test_fr_canonical_check_and_reduction(hk):
    out = ctypes.create_string_buffer(32)
    for v in EDGE + [R, R + 1, (1 << 255) - 1, 1 << 255, (1 << 256) - 1, 2 * R, 2 * R - 1, 3 * R - 1 if 3 * R < (1 << 256) else R]:
        ok = hk.hk_fr_from_be32(_be(v), out)
        assert ok == (v < R), hex(v)
        if ok:
            assert int.from_bytes(out.raw, "big") == v
        hk.hk_fr_reduce(_be(v), out)
        assert int.from_bytes(out.raw, "big") == v % R, hex(v)


def test_roots_of_unity_bit_reversed(hk):
    out = ctypes.create_string_buffer(32)
    for i in list(range(16)) + [1000, 2048, 4095]:
        hk.hk_root_brp(i, out)
        assert int.from_bytes(out.raw, "big") == ko.ROOTS_BRP[i], i
    assert pow(ko.OMEGA, 4096, R) == 1 and pow(ko.OMEGA, 2048, R) != 1


@pytest.mark.parametrize("parts", [1, 256])
def test_evaluation_against_oracle(hk, parts):
    rng = random.Random(7 + parts)
    poly = [rng.randrange(R) for _ in range(4096)]
    blob = b"".join(_be(v) for v in poly)
    out = ctypes.create_string_buffer(32)
    z = rng.randrange(R)
    assert hk.hk_eval(blob, _be(z), parts, out) == 0
    assert int.from_bytes(out.raw, "big") == ko.evaluate_polynomial_in_evaluation_form(poly, z)
    # z forced into the domain: the spec's in-domain branch returns the element at that position
    for i in (0, 1, 2049, 4095):
        assert hk.hk_eval(blob, _be(ko.ROOTS_BRP[i]), parts, out) == 0
        assert int.from_bytes(out.raw, "big") == poly[i] == ko.evaluate_polynomial_in_evaluation_form(poly, ko.ROOTS_BRP[i])
    # an element >= r
    bad = bytearray(blob)
    bad[32 * 100:32 * 101] = _be(R)
    assert hk.hk_eval(bytes(bad), _be(z), parts, out) == 17
