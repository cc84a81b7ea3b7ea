"""chacha20.cuh built for the host: the ChaCha20 block function matches RFC 8439, and the coefficients k_rlc_rho
expands from a seed land where k_rlc_prepare reads them (16 B per proof, 64-bit halves rho_1 and rho_2)."""
import ctypes as C
import os
import struct
import subprocess

import pytest

from conftest import ROOT

U32 = 0xFFFFFFFF


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = tmp_path_factory.mktemp("chacha") / "chacha_host.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                    os.path.join(ROOT, "tests", "host_shim", "chacha_host.cpp")], check=True)
    return C.CDLL(str(out))


def words(b):
    return (C.c_uint32 * (len(b) // 4))(*struct.unpack(f"<{len(b) // 4}I", b))


def block(shim, key, counter, nonce):
    out = (C.c_uint32 * 16)()
    shim.chacha20_block_host(words(key), C.c_uint32(counter), words(nonce), out)
    return struct.pack("<16I", *out)


def py_block(key, counter, nonce):
    """RFC 8439 §2.3 in Python: an independent statement of the block function."""
    def rotl(v, c):
        return ((v << c) | (v >> (32 - c))) & U32

    def qr(x, a, b, c, d):
        x[a] = (x[a] + x[b]) & U32; x[d] = rotl(x[d] ^ x[a], 16)
        x[c] = (x[c] + x[d]) & U32; x[b] = rotl(x[b] ^ x[c], 12)
        x[a] = (x[a] + x[b]) & U32; x[d] = rotl(x[d] ^ x[a], 8)
        x[c] = (x[c] + x[d]) & U32; x[b] = rotl(x[b] ^ x[c], 7)

    s = [0x61707865, 0x3320646E, 0x79622D32, 0x6B206574, *struct.unpack("<8I", key), counter, *struct.unpack("<3I", nonce)]
    x = list(s)
    for _ in range(10):
        qr(x, 0, 4, 8, 12); qr(x, 1, 5, 9, 13); qr(x, 2, 6, 10, 14); qr(x, 3, 7, 11, 15)
        qr(x, 0, 5, 10, 15); qr(x, 1, 6, 11, 12); qr(x, 2, 7, 8, 13); qr(x, 3, 4, 9, 14)
    return struct.pack("<16I", *[(a + b) & U32 for a, b in zip(x, s)])


def test_block_function_matches_rfc8439(shim):
    # RFC 8439 §2.3.2: key 00 01 .. 1f, block counter 1, nonce 00 00 00 09 00 00 00 4a 00 00 00 00
    key = bytes(range(32))
    nonce = bytes.fromhex("000000090000004a00000000")
    want = bytes.fromhex(
        "10f1e7e4d13b5915500fdd1fa32071c4c7d1f4c733c068030422aa9ac3d46c4e"
        "d2826446079faa0914c2d705d98b02a2b5129cd1de164eb9cbd083e8a2503c4e")
    assert block(shim, key, 1, nonce) == want
    assert py_block(key, 1, nonce) == want
    for k in range(4):                                                  # other keys and counters, incl. the wrap of word 12
        key = bytes((7 * k + 13 * i) & 0xFF for i in range(32))
        for ctr in (0, 5, U32):
            assert block(shim, key, ctr, bytes(12)) == py_block(key, ctr, bytes(12)), (k, ctr)


def test_rho_layout_is_what_the_per_proof_kernel_reads(shim):
    # k_rlc_prepare reads proof p's coefficient as the uint4 at rho + 16 p: k[0..3], rho_1 = k0 | k1 << 32 and
    # rho_2 = k2 | k3 << 32 (ec.cuh scalar_mul_glv64).  Proofs 2 and 9 sit in blocks 0 and 2, at quarters 2 and 1.
    seed = bytes((31 * i + 5) & 0xFF for i in range(32))
    n = 11                                                               # the last block is partial
    rho = (C.c_uint32 * (4 * n + 4))(*([0xDEADBEEF] * (4 * n + 4)))
    shim.rlc_rho_host(words(seed), C.c_uint32(n), rho)
    raw = struct.pack(f"<{4 * n + 4}I", *rho)
    for p in (2, 9):
        blk = py_block(seed, p // 4, bytes(12))
        k = struct.unpack("<4I", raw[16 * p:16 * p + 16])
        rho1, rho2 = k[0] | k[1] << 32, k[2] | k[3] << 32
        assert rho1 == int.from_bytes(blk[16 * (p % 4):16 * (p % 4) + 8], "little"), p
        assert rho2 == int.from_bytes(blk[16 * (p % 4) + 8:16 * (p % 4) + 16], "little"), p
    for p in range(n):                                                   # every proof: its quarter of its block
        assert raw[16 * p:16 * p + 16] == py_block(seed, p // 4, bytes(12))[16 * (p % 4):16 * (p % 4) + 16], p
    assert raw[16 * n:] == struct.pack("<4I", *([0xDEADBEEF] * 4))       # nothing written past proof n - 1
