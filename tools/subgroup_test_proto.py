"""Big-integer check of the BN254 G2 membership test the device uses (Dai, Lin, Zhao, Zhou, "Fast subgroup membership
testings for G1, G2 and GT on pairing-friendly curves", ePrint 2022/348, sec. 3 and 5.1; the form gnark-crypto ships):
    P in G2  <=>  [x+1]P + psi([x]P) + psi^2([x]P) == psi^3([2x]P),        x = 4965661367192848881,
one 63-bit scalar multiplication instead of the 127-bit [6x^2]P == psi(P).  Ground truth here: [r]T == O."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import pairing_proto as pp
from pairing_proto import O, f2mul, f2conj, f2sqr, f2add, f2pow, TW_X, TW_Y, B_TWIST, BN_X, P, R, F2_ONE

psi = lambda T: None if T is None else (f2mul(f2conj(T[0]), TW_X), f2mul(f2conj(T[1]), TW_Y))
G2 = O.G2


def fast_test(T):
    a = G2.mul(T, BN_X)
    b = psi(a)
    a1 = G2.add(a, T)
    c = psi(b)
    lhs = G2.add(G2.add(a1, b), c)
    rhs = psi(c)
    rhs = G2.add(rhs, rhs)
    return lhs == rhs


def old_test(T):
    return psi(T) == G2.mul(T, 6 * BN_X * BN_X)


def f2sqrt(a):
    a1 = f2pow(a, (P - 3) // 4)
    alpha = f2mul(a1, f2mul(a1, a))
    x0 = f2mul(a1, a)
    if alpha == ((-1) % P, 0):
        x = f2mul((0, 1), x0)
    else:
        x = f2mul(f2pow(f2add(F2_ONE, alpha), (P - 1) // 2), x0)
    return x if f2sqr(x) == a else None


def main():
    n_in = n_out = 0
    for k in (1, 2, 3, 12345, R - 1, 0x1234567890abcdef1234567890abcdef):
        T = G2.mul(O.G2_GEN, k)
        assert fast_test(T) and old_test(T)
        n_in += 1
    S = G2.mul(O.G2_GEN, 777)
    for t in range(1, 400):
        xx = (t, 1)
        y = f2sqrt(f2add(f2mul(f2sqr(xx), xx), B_TWIST))
        if y is None:
            continue
        T = (xx, y)
        for U in (T, G2.add(T, S), G2.mul(T, R), G2.mul(T, 10069)):      # raw, shifted by a subgroup point, pure cofactor part, a multiple
            if U is None:
                continue
            truth = G2.mul(U, R) is None
            assert fast_test(U) == truth and old_test(U) == truth, (t, truth)
            n_in += truth
            n_out += (not truth)
        if n_out >= 60:
            break
    print("fast G2 membership test agrees with [r]T == O on", n_in, "subgroup points and", n_out, "points outside it")


if __name__ == "__main__":
    main()
