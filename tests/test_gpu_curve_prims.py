"""ec.cuh on the device (the sm_100a build of tests/device_shim/prim_ops.h): the G1 and G2 group law (madd, add,
add_cold, dbl, dbl_affine, from_affine, to_affine, neg, G1's madd_lazy), the ladders (scalar_mul_window at 254 and 128
bits, joint_mul_u128 with phi / psi as rerandomize.cu runs it, scalar_mul_glv64), gather_point's sign handling, and the
scalar splits and window recodings, on the crafted cases of test_curve_prims_host.py.  Every device output must equal
the host build's bit for bit, and then the big-integer oracle."""
import numpy as np
import pytest

import prim_shim as ps
from test_curve_prims_host import Group, all_curve_cases, chain_check, scalar_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev(tmp_path_factory):
    return ps.device(tmp_path_factory)


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return ps.host(tmp_path_factory)


def both(dev, host, fam, code, rec):
    """device output, after requiring it to equal the host build's bit for bit"""
    d, h = dev.run(fam, code, rec), host.run(fam, code, rec)
    bad = np.flatnonzero((d != h).any(axis=1))
    assert bad.size == 0, (fam, code, "device != host build", bad[:5].tolist())
    return d


def test_group_law_and_ladders(dev, host, po):
    for name, fam, code, rec, check in all_curve_cases(po, 131):
        out = both(dev, host, fam, code, rec)
        check(out)


@pytest.mark.parametrize("g, lazy", [(1, False), (1, True), (2, False)], ids=["g1", "g1_lazy", "g2"])
def test_madd_chains_through_infinity(dev, host, po, g, lazy):
    run = lambda fam, code, rec: both(dev, host, fam, code, rec)
    chain_check(Group(po, g), run, 17 + g, steps=300 if g == 1 else 120, chains=32 if g == 1 else 4, lazy=lazy)


def test_splits_and_recoding(dev, host):
    for name, code, rec, check in scalar_cases():
        check(both(dev, host, ps.FAM_SCALAR, code, rec))
