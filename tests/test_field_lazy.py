"""CPU tier: lazy-reduction field arithmetic (fp.cuh mul_wide / sqr_wide / redc / sqr / mul_sub, fp2.cuh mul / sqr /
mul_sub) and the XYZZ formulas built on it, stepped on the host by a plain C++ build of the device headers
(tests/host_emu/emu_field_lazy.cpp, -DZKB_EMU) and checked against Python big-int arithmetic.

Field operations are checked on raw limb values: every result must be the canonical residue (ab - cd) R^-1 mod p,
including the bound cases (operands p - 1, redc of p R - 1, results 0 and p - 1)."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from oracle.ff import BLS12_381, BN254, g1_group, g2_group

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "zokrates_b200", "csrc")
HARNESS = os.path.join(ROOT, "tests", "host_emu", "emu_field_lazy.cpp")

# (harness field id, modulus, limbs)
FIELDS = {"bn254_fr": (0, BN254.r, 8), "bn254_fq": (1, BN254.p, 8), "bls12_381_fr": (2, BLS12_381.r, 8),
          "bls12_381_fq": (3, BLS12_381.p, 12)}
CURVES = [(0, BN254, 8), (1, BLS12_381, 12)]
RANDOM_CASES = 10_000


@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("lazy") / "emu_field_lazy.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-DZKB_EMU", "-shared", "-fPIC", "-I", CSRC, HARNESS, "-o", out], check=True)
    dll = C.CDLL(out)
    dll.emu_lazy_fp.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    dll.emu_lazy_fp2.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    dll.emu_lazy_ec.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int]
    return dll


def pack(values, nl):
    """ints -> little-endian 32-bit limbs, nl limbs each, back to back"""
    return np.frombuffer(b"".join(int(v).to_bytes(4 * nl, "little") for v in values), dtype=np.uint32).copy()


def unpack(words, nl):
    b = words.tobytes()
    return [int.from_bytes(b[4 * nl * i:4 * nl * (i + 1)], "little") for i in range(len(words) // nl)]


def run(fn, args, values, nl_in, n, nl_out, per=1):
    """n cases; each returns `per` values of nl_out limbs"""
    inp = pack(values, nl_in)
    out = np.zeros(n * per * nl_out, dtype=np.uint32)
    fn(*args, inp.ctypes.data, out.ctypes.data, n)
    return unpack(out, nl_out)


def fp_cases(p, R, rnd):
    """(a, b, c, d) quadruples: bound cases first, then random ones"""
    m = p - 1
    a, b = rnd.randrange(1, p), rnd.randrange(1, p)
    c = rnd.randrange(1, p)
    cases = [(m, m, m, m), (m, m, 0, 0), (0, 0, m, m), (0, 0, 0, 0), (1, 1, 1, 1),
             (a, b, a, b), (a, b, b, a),                          # a b = c d: result 0
             (a, b, c, (a * b + R) * pow(c, -1, p) % p),          # result -R R^-1 = p - 1
             (m, 1, 0, 0), (1, m, m, 1)]
    cases += [tuple(rnd.randrange(p) for _ in range(4)) for _ in range(RANDOM_CASES)]
    return cases


@pytest.mark.parametrize("name", list(FIELDS))
def test_fp_lazy_ops(lib, name):
    fid, p, nl = FIELDS[name]
    R = 1 << (32 * nl)
    Ri = pow(R, -1, p)
    rnd = random.Random(fid)
    cases = fp_cases(p, R, rnd)
    n = len(cases)
    flat = [v for q in cases for v in q]
    a = [q[0] for q in cases]
    ab = [v for q in cases for v in q[:2]]
    assert run(lib.emu_lazy_fp, (fid, 1), flat, nl, n, nl) == [(x * y - z * w) * Ri % p for x, y, z, w in cases]
    assert run(lib.emu_lazy_fp, (fid, 0), a, nl, n, nl) == [x * x * Ri % p for x in a]
    assert run(lib.emu_lazy_fp, (fid, 2), ab, nl, n, 2 * nl) == [x * y for x, y, _, _ in cases]
    assert run(lib.emu_lazy_fp, (fid, 3), a, nl, n, 2 * nl) == [x * x for x in a]
    # sqr_wide / mul_wide take any N-limb operand, e.g. the unreduced sums (< 2p) of the Fq2 Karatsuba, and all-ones limbs
    wide_ops = [R - 1, 2 * p - 1, 2 * p - 2] + [rnd.randrange(2 * p) for _ in range(200)]
    assert run(lib.emu_lazy_fp, (fid, 3), wide_ops, nl, len(wide_ops), 2 * nl) == [x * x for x in wide_ops]
    # redc: any T < p R, up to the bound itself
    T = [0, 1, p * R - 1, p * R - R, p * p, 2 * p * p - 1, (p - 1) * (p - 1)] + [rnd.randrange(p * R) for _ in range(RANDOM_CASES)]
    assert run(lib.emu_lazy_fp, (fid, 4), T, 2 * nl, len(T), nl) == [t * Ri % p for t in T]


def fp2_mul(p, x, y):
    return ((x[0] * y[0] - x[1] * y[1]) % p, (x[0] * y[1] + x[1] * y[0]) % p)


@pytest.mark.parametrize("cid,c,nl", CURVES, ids=[c.name for _, c, _ in CURVES])
def test_fp2_lazy_ops(lib, cid, c, nl):
    p = c.p
    R = 1 << (32 * nl)
    Ri = pow(R, -1, p)
    rnd = random.Random(10 + cid)
    m = p - 1
    el = lambda: (rnd.randrange(p), rnd.randrange(p))
    a, b, cc = el(), el(), el()
    ab = fp2_mul(p, a, b)
    # d with c d = a b + R (u + 1): result (p - 1, p - 1)
    cn = (cc[0] * cc[0] + cc[1] * cc[1]) % p
    cinv = (cc[0] * pow(cn, -1, p) % p, -cc[1] * pow(cn, -1, p) % p)
    d_m1 = fp2_mul(p, ((ab[0] + R) % p, (ab[1] + R) % p), cinv)
    mm, z = (m, m), (0, 0)
    cases = [(mm, mm, mm, mm), (mm, mm, z, z), (z, z, mm, mm), ((m, 0), (0, m), (0, m), (m, 0)), ((0, m), (0, m), (m, 0), (m, 0)),
             (a, b, a, b), (a, b, b, a), (a, b, cc, d_m1), (z, z, z, z)]
    cases += [(el(), el(), el(), el()) for _ in range(RANDOM_CASES)]
    n = len(cases)
    scale = lambda v: (v[0] * Ri % p, v[1] * Ri % p)
    got = run(lib.emu_lazy_fp2, (cid, 2), [x for q in cases for e in q for x in e], nl, n, nl, 2)
    want = []
    for q in cases:
        u, v = fp2_mul(p, q[0], q[1]), fp2_mul(p, q[2], q[3])
        want += scale(((u[0] - v[0]) % p, (u[1] - v[1]) % p))
    assert got == want
    assert (m, m) == tuple(got[14:16])                         # the case built to land on p - 1
    got = run(lib.emu_lazy_fp2, (cid, 0), [x for q in cases for e in q[:2] for x in e], nl, n, nl, 2)
    assert got == [x for q in cases for x in scale(fp2_mul(p, q[0], q[1]))]
    got = run(lib.emu_lazy_fp2, (cid, 1), [x for q in cases for x in q[0]], nl, n, nl, 2)
    assert got == [x for q in cases for x in scale(fp2_mul(p, q[0], q[0]))]


# ---- XYZZ formulas against the affine group law ------------------------------------------------------------------


class Enc:
    """Montgomery limb encoding of G1 / G2 points for one curve."""

    def __init__(self, c, nl, group):
        self.c, self.nl, self.g2 = c, nl, group == 2
        self.p = c.p
        self.R = 1 << (32 * nl)
        self.G = g2_group(c) if self.g2 else g1_group(c)
        self.F = self.G.F
        self.k = 2 if self.g2 else 1                          # base-field elements per coordinate

    def coord(self, v):
        v = v if self.g2 else (v,)
        return [x * self.R % self.p for x in v]

    def affine(self, P):
        return self.coord(self.F.zero) * 2 if P is None else self.coord(P[0]) + self.coord(P[1])

    def xyzz(self, P, z):
        F = self.F
        if P is None:
            return self.coord(F.zero) * 4
        zz = F.sqr(z)
        zzz = F.mul(zz, z)
        return self.coord(F.mul(P[0], zz)) + self.coord(F.mul(P[1], zzz)) + self.coord(zz) + self.coord(zzz)

    def decode(self, limbs):
        """XYZZ limbs -> affine point (None: identity); every output word must be canonical (< p)"""
        assert all(0 <= v < self.p for v in limbs)
        Ri = pow(self.R, -1, self.p)
        vals = [v * Ri % self.p for v in limbs]
        co = [tuple(vals[i:i + 2]) if self.g2 else vals[i] for i in range(0, 4 * self.k, self.k)]
        X, Y, ZZ, ZZZ = co
        F = self.F
        if F.is_zero(ZZ):
            return None
        assert F.mul(F.sqr(ZZ), ZZ) == F.sqr(ZZZ)               # ZZ^3 = ZZZ^2
        return (F.mul(X, F.inv(ZZ)), F.mul(Y, F.inv(ZZZ)))


def rand_z(F, rnd, p):
    return (rnd.randrange(1, p), rnd.randrange(p)) if isinstance(F.zero, tuple) else rnd.randrange(1, p)


@pytest.mark.parametrize("group", [1, 2], ids=["g1", "g2"])
@pytest.mark.parametrize("cid,c,nl", CURVES, ids=[c.name for _, c, _ in CURVES])
def test_xyzz_formulas(lib, cid, c, nl, group):
    e = Enc(c, nl, group)
    G, F = e.G, e.F
    rnd = random.Random(100 * cid + group)
    gen = c.g2 if group == 2 else c.g1
    pts = [G.mul(gen, rnd.randrange(1, c.r)) for _ in range(6)]
    P, Q, S = pts[0], pts[1], pts[2]
    z = lambda: rand_z(F, rnd, c.p)
    one = F.one

    def call(op, n, words):
        return run(lambda *a: lib.emu_lazy_ec(cid, group, *a), (op,), words, nl, n, nl, 4 * e.k)

    def check(op, cases, inputs, want):
        got = call(op, len(cases), [w for x in inputs for w in x])
        assert [e.decode(got[i * 4 * e.k:(i + 1) * 4 * e.k]) for i in range(len(cases))] == want

    # madd: generic, P + P (doubling branch), P + (-P), identity accumulator, point at infinity, accumulator with Z = 1
    madd = [(P, z(), Q), (S, z(), P), (P, z(), P), (Q, one, Q), (P, z(), G.neg(P)), (None, one, Q), (P, z(), None),
            (None, one, None), (pts[3], one, pts[4])]
    madd += [(pts[rnd.randrange(6)], z(), pts[rnd.randrange(6)]) for _ in range(8)]
    check(0, madd, [e.xyzz(a, za) + e.affine(q) for a, za, q in madd], [G.add(a, q) for a, za, q in madd])
    # add: generic, P + P, P + (-P), identity on either side, both identity
    add = [(P, z(), Q, z()), (P, z(), P, z()), (P, z(), G.neg(P), z()), (None, one, Q, z()), (Q, z(), None, one),
           (None, one, None, one), (S, one, S, one)]
    add += [(pts[rnd.randrange(6)], z(), pts[rnd.randrange(6)], z()) for _ in range(8)]
    check(1, add, [e.xyzz(a, za) + e.xyzz(b, zb) for a, za, b, zb in add], [G.add(a, b) for a, za, b, zb in add])
    # dbl / mdbl
    dbl = [(P, z()), (Q, one), (None, one)] + [(pts[i], z()) for i in range(3, 6)]
    check(2, dbl, [e.xyzz(a, za) for a, za in dbl], [G.add(a, a) for a, za in dbl])
    mdbl = pts
    check(3, mdbl, [e.affine(a) for a in mdbl], [G.add(a, a) for a in mdbl])
