"""Proof rerandomization on the host: ec.cuh psi_split built with g++ splits exactly, the oracle's psi is [6 x^2] on G2,
rerandomized oracle proofs still verify and compose, and rerandomize.cu compiles for sm_100a."""
import ctypes as C
import os
import random
import shutil
import subprocess

import pytest

from conftest import ROOT
from oracle import zkp_rerandomize as zr

R = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
L = zr.LAMBDA_PSI


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = tmp_path_factory.mktemp("psi") / "psi_split_host.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                    os.path.join(ROOT, "tests", "host_shim", "psi_split_host.cpp")], check=True)
    return C.CDLL(str(out))


def split(shim, ks):
    n = len(ks)
    k = (C.c_uint32 * (8 * n))(*[(v >> (32 * j)) & 0xFFFFFFFF for v in ks for j in range(8)])
    k0, k1 = (C.c_uint32 * (4 * n))(), (C.c_uint32 * (4 * n))()
    shim.psi_split_host(k, k0, k1, n)
    join = lambda a, i: sum(a[4 * i + j] << (32 * j) for j in range(4))
    return [(join(k0, i), join(k1, i)) for i in range(n)]


def test_lambda_psi():
    assert L == 0x6F4D8248EEB859FBF83E9682E87CFD46 and L < R and L.bit_length() == 127


def test_psi_split_exact(shim):
    edges = [0, 1, 2, L - 1, L, L + 1, R - 1, R - 2, R - L, R - L - 1]
    for m in (2, 3, 7, (R - 1) // L - 1, (R - 1) // L):
        edges += [m * L - 1, m * L, m * L + 1]
    rng = random.Random(20201811)
    ks = [k for k in edges if 0 <= k < R] + [rng.randrange(R) for _ in range(100_000)]
    for k, (k0, k1) in zip(ks, split(shim, ks)):
        assert (k0, k1) == (k % L, k // L), hex(k)
        assert k0 + k1 * L == k and k0 < 2 ** 128 and k1 < 2 ** 128


def test_psi_is_lambda_psi(po):
    rng = po.SplitMix64(41)
    for _ in range(3):
        Q = po.G2.mul(po.G2_GEN, rng.next_fr())
        assert zr.psi(Q) == po.G2.mul(Q, L)
        assert zr.psi(po.G2.add(Q, po.G2_GEN)) == po.G2.add(zr.psi(Q), zr.psi(po.G2_GEN))
    assert zr.psi(None) is None


def test_rerandomized_proofs_verify_and_compose(po, golden):
    case = golden["equality"]["proofs"][0]
    vk = po.vk_from_bytes(bytes.fromhex(golden["equality"]["vk"]))
    proof = po.proof_from_bytes(bytes.fromhex(case["proof"]))
    x = po.equality_public_inputs(int.from_bytes(po.commit_value_snark(case["a"]), "little"))
    assert po.verify(vk, x, proof)
    r1, r2, s1, s2 = 0x1234567, R - 5, 0xABCDEF0123, 3
    p1 = zr.rerandomize(vk.delta_g2, proof, r1, r2)
    assert p1 != proof and all(a != b for a, b in zip(p1, proof))
    assert po.verify(vk, x, p1)
    p2 = zr.rerandomize(vk.delta_g2, p1, s1, s2)
    once = zr.rerandomize(vk.delta_g2, proof, r1 * s1 % R, (r2 + s2 * pow(r1, -1, R)) % R)
    assert p2 == once


def test_checker_bytes_of_rejected_rows(po, golden):
    row = bytes.fromhex(golden["equality"]["proofs"][0]["proof"])
    delta = po.G2_GEN
    assert zr.rerandomize_bytes(delta, row, 0, 1) == b"\xff" * 256
    assert zr.rerandomize_bytes(delta, row, 1, R) == b"\xff" * 256
    both = bytearray(row)
    both[63] |= 0xC0
    assert zr.rerandomize_bytes(delta, bytes(both), 1, 1) == b"\xff" * 256
    assert zr.rerandomize_bytes(delta, row, 1, 1) != b"\xff" * 256


@pytest.mark.skipif(shutil.which("nvcc") is None and not os.path.exists("/usr/local/cuda/bin/nvcc"), reason="no nvcc")
def test_rerandomize_cu_compiles_for_sm100a(tmp_path):
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    src = os.path.join(ROOT, "libzkp_b200", "csrc", "rerandomize.cu")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-Xcompiler", "-fPIC",
                    "-c", src, "-o", str(tmp_path / "rerandomize.o")], check=True)
