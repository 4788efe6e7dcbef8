"""The product's FarmHash (csrc/farmhash.cuh, the __host__ __device__ code the fingerprint / hash-partition kernels run,
compiled for the host inside libytgpu.so) against the REFERENCE'S OWN contrib/libs/farmhash/farmhash.cc — no restatement
in between: against its outputs stored in tests/golden/farmhash_reference.json, and against its build
(oracle/_ref/libfarmhash_ref.so) as well where oracle.build() found a YTsaurus source tree."""
import ctypes as C
import hashlib
import json
import os

import pytest

import oracle
from ytsaurus_b200 import capi

GOLDEN = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "farmhash_reference.json")))
LENGTHS = [0, 1, 3, 4, 7, 8, 16, 17, 32, 33, 63, 64, 65, 127, 128, 129, 191, 192, 193, 1023, 1024, 1025, 65536, 1 << 20]


def _product():
    lib = capi.load()
    lib.ytgpu_hostcheck_fingerprint_bytes.restype = C.c_uint64
    lib.ytgpu_hostcheck_fingerprint_bytes.argtypes = [C.c_char_p, C.c_uint64]
    return lib


def _check(data, want):
    assert _product().ytgpu_hostcheck_fingerprint_bytes(data, len(data)) == want, len(data)
    if oracle.ref_lib() is not None:
        assert oracle.ref_lib().ref_fingerprint64(data, len(data)) == want, len(data)


def test_fingerprint_of_any_byte_string():
    # 1500 seeded byte strings, every length 0..400 three or four times
    for i, want in enumerate(GOLDEN["any_byte_string"]):
        _check(hashlib.shake_128(f"any {i}".encode()).digest(i % 401), int(want))


@pytest.mark.parametrize("n", LENGTHS)
def test_fingerprint_length_classes(n):
    data = bytes((i * 131 + 7) & 0xFF for i in range(n))
    _check(data, int(GOLDEN["length_classes"][str(n)]))
