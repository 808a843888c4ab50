"""featurebase_b200/csrc/stripe.h (experimental bank-striped array payload order, FBGPU_ARRAY_STRIPED=1): the
permutation must be a bijection for every cardinality and never write outside [0, n); on uniform data it must cut the
shared-memory wavefront count of the scatter instruction groups it is modelled on."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("stripe") / "libstripe_check.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(ROOT, "featurebase_b200", "csrc"),
                           os.path.join(ROOT, "tests", "native", "stripe_check.cpp"), "-o", out])
    L = C.CDLL(out)
    # pointers must be declared: ctypes passes an undeclared Python int as a 32-bit C int
    vp, u32 = C.c_void_p, C.c_uint32
    L.stripe.argtypes = [vp, vp, u32]
    L.wavefronts.argtypes, L.wavefronts.restype = [vp, u32], C.c_uint64
    L.worst.argtypes, L.worst.restype = [vp, u32], C.c_uint32
    L.word_offset_mismatches.argtypes, L.word_offset_mismatches.restype = [], C.c_uint64
    L.load_array.argtypes = [vp, vp, u32, C.c_int]
    L.model_scatter.argtypes = [C.c_int, vp, u32, vp]
    L.model_probe.argtypes = [vp, u32, vp]
    return L


def _stripe(L, v):
    d = np.full(len(v) + 8, 0xDEAD, dtype=np.uint16)
    L.stripe(v.ctypes.data, d.ctypes.data, len(v))
    assert (d[len(v):] == 0xDEAD).all()
    return d[: len(v)].copy()


def test_bijection_all_shapes(lib):
    rng = np.random.default_rng(5)
    sizes = list(range(0, 70)) + [100, 255, 256, 257, 511, 512, 513, 655, 1000, 2047, 2048, 4000, 4095]
    for n in sizes:
        for kind in range(4):
            if kind == 0:
                v = np.sort(rng.choice(65536, n, replace=False)).astype(np.uint16)
            elif kind == 1:
                v = (np.arange(n) + 777).astype(np.uint16)                       # one dense block: few banks per group
            elif kind == 2:
                v = np.sort(((np.arange(n) % 64) * 1024 + np.arange(n) // 64)).astype(np.uint16)    # every element in bank 0/1
            else:
                v = np.sort(rng.choice(4096, min(n, 4096), replace=False) * 16).astype(np.uint16)   # clustered
            v = np.ascontiguousarray(v)
            d = _stripe(lib, v)
            assert np.array_equal(np.sort(d), v), (n, kind)


def test_unaligned_source(lib):
    rng = np.random.default_rng(6)
    v = np.sort(rng.choice(65536, 700, replace=False)).astype(np.uint16)
    raw = np.zeros(2 * len(v) + 1, dtype=np.uint8)
    raw[1:] = v.view(np.uint8)                                                   # odd address, as inside a roaring file
    d = np.zeros(len(v), dtype=np.uint16)
    lib.stripe(C.c_void_p(raw.ctypes.data + 1), d.ctypes.data, len(v))
    assert np.array_equal(np.sort(d), v)


def test_wavefront_reduction_uniform(lib):
    rng = np.random.default_rng(7)
    before = after = ideal = 0
    for _ in range(200):
        n = int(rng.integers(500, 800))                                          # ~1 % density containers (BASELINE configs)
        v = np.ascontiguousarray(np.sort(rng.choice(65536, n, replace=False)).astype(np.uint16))
        d = _stripe(lib, v)
        before += lib.wavefronts(v.ctypes.data, n)
        after += lib.wavefronts(d.ctypes.data, n)
        ideal += 8 * (n // 256) + min(8, n % 256)
    assert after < 0.45 * before          # measured here: ~0.37
    assert after < 1.35 * ideal


def test_word_offset_identity(lib):
    """csrc/bitaddr.h: 4 * (element >> 5) written as mask + multiply-high (so that ptxas emits LOP3 + LEA.HI) equals the
    plain form for every lower element and a spread of upper elements, and vice versa"""
    assert lib.word_offset_mismatches() == 0


def test_array_tail_padding(lib):
    """the slots behind the last element of a stored array repeat a VALID element (never a zero that would set bit 0):
    the OR / AND-NOT scatter runs whole 16-byte chunks unguarded"""
    rng = np.random.default_rng(9)
    for n in list(range(1, 40)) + [63, 64, 65, 655, 4079, 4090, 4095, 4096]:
        for striped in (0, 1):
            v = np.ascontiguousarray(np.sort(rng.choice(np.arange(1, 65536), n, replace=False)).astype(np.uint16))    # 0 is absent on purpose
            padded = (n + 7) & ~7
            d = np.full(padded + 8, 0xDEAD, dtype=np.uint16)
            lib.load_array(v.ctypes.data, d.ctypes.data, n, striped)
            assert (d[padded:] == 0xDEAD).all()
            assert np.array_equal(np.sort(d[:n]), v)
            assert set(d[n:padded].tolist()) <= {int(d[n - 1])}
            assert set(np.unique(d[:padded]).tolist()) == set(v.tolist())          # the chunked bit set is exactly the container


def test_scatter_and_probe_model_on_stored_payloads(lib):
    """host model of scatter_chunk_sb / probe_chunk (same helper headers, same control flow) over payloads exactly as the
    loader stores them (plain or striped order, duplicate-padded tail): OR sets exactly the container, AND-NOT clears
    exactly it, XOR toggles exactly it, and the probe counts exactly the intersection — for every tail length"""
    rng = np.random.default_rng(10)
    lib.model_probe.restype = C.c_uint32
    for n in list(range(1, 34)) + [63, 64, 65, 100, 655, 1000, 4079, 4095, 4096]:
        for striped in (0, 1):
            v = np.ascontiguousarray(np.sort(rng.choice(65536, n, replace=False)).astype(np.uint16))
            padded = (n + 7) & ~7
            pay = np.zeros(padded, dtype=np.uint16)
            lib.load_array(v.ctypes.data, pay.ctypes.data, n, striped)
            want = np.zeros(65536, dtype=bool)
            want[v] = True
            other = rng.random(65536) < 0.3
            def bits(words):
                return np.unpackbits(words.view(np.uint8), bitorder="little").astype(bool)
            def words(mask):
                return np.packbits(mask, bitorder="little").view(np.uint32).copy()
            bm = words(other)
            lib.model_scatter(0, pay.ctypes.data, n, bm.ctypes.data)
            assert np.array_equal(bits(bm), other | want), (n, striped, "or")
            bm = words(other)
            lib.model_scatter(1, pay.ctypes.data, n, bm.ctypes.data)
            assert np.array_equal(bits(bm), other & ~want), (n, striped, "andnot")
            bm = words(other)
            lib.model_scatter(2, pay.ctypes.data, n, bm.ctypes.data)
            assert np.array_equal(bits(bm), other ^ want), (n, striped, "xor")
            bm = words(other)
            assert lib.model_probe(pay.ctypes.data, n, bm.ctypes.data) == int((other & want).sum()), (n, striped, "probe")
