"""ark-serialize's compressed form on the host: the oracle's compressed encode / decode round-trips, and the engine's
host-side compression (lzkp_pk_compress, lzkp_vk_compress, lzkp_proofs_compress) is byte-equal to the oracle's
compressed encoders on real keys and golden proofs, and refuses malformed input."""
import ctypes as C

import numpy as np
import pytest

from conftest import has_gpu

from libzkp_b200 import _ffi, engine
from libzkp_b200.errors import EngineError
from oracle import zkp_compressed as pc


def _points(po, seed, n):
    rng = po.SplitMix64(seed)
    ks = [rng.next_fr() for _ in range(n)]
    return [po.G1.mul(po.G1_GEN, k) for k in ks], [po.G2.mul(po.G2_GEN, k) for k in ks]


def test_oracle_round_trip(po):
    g1, g2 = _points(po, 11, 12)
    signs1, signs2 = set(), set()
    for P in g1 + [po.G1.neg(P) for P in g1]:
        b = pc.g1_to_bytes_compressed(P)
        assert len(b) == 32 and pc.g1_from_bytes_compressed(b) == P
        assert b[:31] == po.g1_to_bytes(P)[:31] and (b[31] & 0x80) == (po.g1_to_bytes(P)[63] & 0x80)
        signs1.add(b[31] >> 7)
    for Q in g2 + [po.G2.neg(Q) for Q in g2]:
        b = pc.g2_to_bytes_compressed(Q)
        assert len(b) == 64 and pc.g2_from_bytes_compressed(b) == Q
        assert (b[63] & 0x80) == (po.g2_to_bytes(Q)[127] & 0x80)
        signs2.add(b[63] >> 7)
    assert signs1 == {0, 1} and signs2 == {0, 1}                       # both roots are exercised
    assert pc.g1_to_bytes_compressed(None) == bytes(31) + b"\x40"
    assert pc.g2_to_bytes_compressed(None) == bytes(63) + b"\x40"
    assert pc.g1_from_bytes_compressed(bytes(31) + b"\x40") is None
    assert pc.g2_from_bytes_compressed(bytes(63) + b"\x40") is None


def test_oracle_rejects_malformed(po):
    g1, g2 = _points(po, 12, 1)
    with pytest.raises(ValueError):                                    # x >= q
        pc.g1_from_bytes_compressed(po.Q_MOD.to_bytes(32, "little"))
    with pytest.raises(ValueError):                                    # both flags
        pc.g1_from_bytes_compressed(bytes(31) + b"\xc0")
    x = next(x for x in range(1, 100) if pc.fq_sqrt(x ** 3 + 3) is None)
    with pytest.raises(ValueError):                                    # x^3 + 3 a non-residue
        pc.g1_from_bytes_compressed(x.to_bytes(32, "little"))
    b = bytearray(pc.g2_to_bytes_compressed(g2[0]))
    b[31] |= 0x80                                                      # flags on x.c0
    with pytest.raises(ValueError):
        pc.g2_from_bytes_compressed(bytes(b))


def test_oracle_object_sizes(po, eq_keys, golden):
    vk = po.vk_from_bytes(eq_keys.vk_bytes)
    n_pub = len(vk.gamma_abc_g1) - 1
    assert len(pc.vk_to_bytes_compressed(vk)) == 232 + 32 * (n_pub + 1)
    pk = po.pk_from_bytes(eq_keys.pk_bytes)
    n1 = 2 + len(pk.a_query) + len(pk.b_g1_query) + len(pk.h_query) + len(pk.l_query)
    n2 = len(pk.b_g2_query)
    assert len(eq_keys.pk_bytes) == len(pc.pk_to_bytes_compressed(pk)) + 32 * (n1 + n_pub + 2) + 64 * (n2 + 3)
    for case in golden["equality"]["proofs"]:
        P = po.proof_from_bytes(bytes.fromhex(case["proof"]))
        assert len(pc.proof_to_bytes_compressed(P)) == 128
        assert pc.proof_from_bytes_compressed(pc.proof_to_bytes_compressed(P)) == P


@pytest.mark.parametrize("which", ["eq", "mb"])
def test_key_compress_equals_oracle(po, eq_keys, mb_keys, which):
    keys = eq_keys if which == "eq" else mb_keys
    pk_c = engine.pk_compress(keys.pk_bytes)
    assert pk_c == pc.pk_to_bytes_compressed(po.pk_from_bytes(keys.pk_bytes))
    vk_c = engine.vk_compress(keys.vk_bytes)
    assert vk_c == pc.vk_to_bytes_compressed(po.vk_from_bytes(keys.vk_bytes))
    # the size query reports the same length without an output buffer
    n = C.c_size_t()
    buf = np.frombuffer(keys.pk_bytes, np.uint8)
    assert _ffi.lib().lzkp_pk_compress(engine._p(buf), buf.size, None, 0, C.byref(n)) == 0
    assert n.value == len(pk_c)
    # a too-small buffer is refused
    out = np.zeros(len(pk_c) - 1, np.uint8)
    assert _ffi.lib().lzkp_pk_compress(engine._p(buf), buf.size, engine._p(out), out.size, C.byref(n)) == _ffi.LZKP_E_INVALID


def test_proofs_compress_equals_oracle(po, golden):
    rows = [bytes.fromhex(c["proof"]) for c in golden["equality"]["proofs"] + golden["membership"]["proofs"]]
    proofs = np.frombuffer(b"".join(rows), np.uint8).reshape(-1, 256)
    out, ok = engine.proofs_compress(proofs)
    assert ok.all()
    for i, r in enumerate(rows):
        assert out[i].tobytes() == pc.proof_to_bytes_compressed(po.proof_from_bytes(r))
    # infinity and both signs of every group (the input's 0x80 bit is not trusted: it is recomputed from y)
    g1, g2 = _points(po, 13, 4)
    extra = [(g1[0], g2[0], po.G1.neg(g1[1])), (None, po.G2.neg(g2[2]), g1[3]), (g1[2], None, None)]
    raw = np.frombuffer(b"".join(po.proof_to_bytes(P) for P in extra), np.uint8).reshape(-1, 256).copy()
    raw[0, 63] ^= 0x80                                                 # a wrong sign bit on A's uncompressed form
    out, ok = engine.proofs_compress(raw)
    assert ok.all()
    for i, P in enumerate(extra):
        assert out[i].tobytes() == pc.proof_to_bytes_compressed(P)


def test_proofs_compress_rejects_malformed(po, golden):
    row = np.frombuffer(bytes.fromhex(golden["equality"]["proofs"][0]["proof"]), np.uint8)
    bad = np.tile(row, (5, 1))
    bad[0, 0:32] = np.frombuffer(po.Q_MOD.to_bytes(32, "little"), np.uint8)     # A.x = q
    bad[1, 31] |= 0x40                                                           # flags on A.x
    bad[2, 127] |= 0xC0                                                          # both flags on B
    bad[3, 255] = 0xFF                                                           # C.y >= q
    out, ok = engine.proofs_compress(bad)
    assert ok.tolist() == [False, False, False, False, True]
    assert (out[:4] == 0xFF).all()
    assert out[4].tobytes() == pc.proof_to_bytes_compressed(po.proof_from_bytes(row.tobytes()))


def test_key_compress_rejects_malformed(eq_keys, po):
    pk = bytearray(eq_keys.pk_bytes)
    for bad in (bytes(pk[:-1]), bytes(pk) + b"\0"):                  # truncated, trailing byte
        with pytest.raises(EngineError) as e:
            engine.pk_compress(bad)
        assert e.value.code == _ffi.LZKP_E_INVALID
    pk[0:32] = po.Q_MOD.to_bytes(32, "little")                         # alpha.x = q
    with pytest.raises(EngineError) as e:
        engine.pk_compress(bytes(pk))
    assert e.value.code == _ffi.LZKP_E_INVALID
    vk = bytearray(eq_keys.vk_bytes)
    vk[448 + 7] = 0xFF                                                 # gamma_abc length overruns the bytes
    with pytest.raises(EngineError) as e:
        engine.vk_compress(bytes(vk))
    assert e.value.code == _ffi.LZKP_E_INVALID


@pytest.mark.skipif(has_gpu(), reason="checks the no-device behaviour")
def test_decompression_needs_a_device(eq_keys):
    with pytest.raises(EngineError) as e:
        engine.proofs_decompress(np.zeros((1, 128), np.uint8))
    assert e.value.code == _ffi.LZKP_E_NO_DEVICE
    with pytest.raises(EngineError) as e:
        engine.VerifyingKey(engine.vk_compress(eq_keys.vk_bytes), compressed=True)
    assert e.value.code == _ffi.LZKP_E_NO_DEVICE
