// Quadratic extension Fq2 = Fq[u]/(u^2 + 1) used by G2 of BN254 and BLS12-381
// (ark-bn254 / ark-bls12-381 0.3.0 Fq2Parameters::NONRESIDUE = -1; SURVEY.md App. C).
// Same static interface as Fp<P> so the curve code is generic over the coordinate field.  The base field B is Fp<P> on the
// device and Fp64<P> (fp64.cuh) in the host tail; both provide the lazy-reduction primitives used here.
#pragma once
#include "fp.cuh"

namespace zkb {

template <class Bt>
struct Fp2T {
  typedef Bt B;
  typedef Fp2T Fp2;
  B c0, c1;

  ZKB_HD static Fp2 zero() { return Fp2{B::zero(), B::zero()}; }
  ZKB_HD static Fp2 one() { return Fp2{B::one(), B::zero()}; }
  ZKB_HD bool is_zero() const { return c0.is_zero() && c1.is_zero(); }
  ZKB_HD bool operator==(const Fp2& o) const { return c0 == o.c0 && c1 == o.c1; }
  ZKB_HD bool operator!=(const Fp2& o) const { return !(*this == o); }
  ZKB_HD static Fp2 add(const Fp2& a, const Fp2& b) { return Fp2{B::add(a.c0, b.c0), B::add(a.c1, b.c1)}; }
  ZKB_HD static Fp2 sub(const Fp2& a, const Fp2& b) { return Fp2{B::sub(a.c0, b.c0), B::sub(a.c1, b.c1)}; }
  ZKB_HD static Fp2 neg(const Fp2& a) { return Fp2{B::neg(a.c0), B::neg(a.c1)}; }
  ZKB_HD static Fp2 dbl(const Fp2& a) { return Fp2{B::dbl(a.c0), B::dbl(a.c1)}; }
  // Karatsuba with lazy reduction: 3 products on 2N limbs and 2 Montgomery reductions (SURVEY.md §8d's M2 = 3 counts
  // full multiplications; this is 5N^2 + 2N wide MADs against 6N^2 + 3N).  Squaring: 2 products, 2 reductions.
  // All three are OUT OF LINE with by-value arguments: ptxas passes the operands in registers (no local-memory traffic),
  // and the G2 mixed addition stays a few calls into small bodies instead of a ~6 500-instruction inlined block that
  // misses the 32 KB instruction cache (`no_instruction` was the top stall of the round-1 G2 accumulate kernel).
  // Bounds (each input of redc must be < p R): a0 + a1 and b0 + b1 stay unreduced (< 2p), so the c1 difference is exactly
  // a0 b1 + a1 b0 < 2p^2 and c0 = a0 b0 + p^2 - a1 b1 < 2p^2, both < p R when 2p < R (Fp::redc asserts it).
  typedef typename B::Wide Wide;
  ZKB_NI static Fp2 mul_v(Fp2 a, Fp2 b) {
    Wide v0 = B::mul_wide(a.c0, b.c0);
    Wide v1 = B::mul_wide(a.c1, b.c1);
    Wide s = B::mul_wide(B::add_raw(a.c0, a.c1), B::add_raw(b.c0, b.c1));
    return Fp2{B::redc(B::sub_wide(B::add_wide(v0, B::p2()), v1)), B::redc(B::sub_wide(B::sub_wide(s, v0), v1))};
  }
  // (a0 + a1)(a0 - a1) < 2p^2 and (2 a0) a1 < 2p^2
  ZKB_NI static Fp2 sqr_v(Fp2 a) {
    return Fp2{B::redc(B::mul_wide(B::add_raw(a.c0, a.c1), B::sub(a.c0, a.c1))), B::redc(B::mul_wide(B::add_raw(a.c0, a.c0), a.c1))};
  }
  // a b - c d: six products, two reductions.  Offset 2p^2 on both components: c0 = a0 b0 - a1 b1 - c0 d0 + c1 d1 + 2p^2 and
  // c1 = (a0 b1 + a1 b0) - (c0 d1 + c1 d0) + 2p^2 lie in (0, 4p^2), < p R when 4p < R; no partial sum exceeds 6p^2 < R^2.
  ZKB_NI static Fp2 mul_sub_v(Fp2 a, Fp2 b, Fp2 c, Fp2 d) {
    static_assert(B::Params::BITS + 2 <= 32 * B::Params::N, "mul_sub_v needs 4p < R");
    Wide im = B::add_wide(B::mul_wide(B::add_raw(a.c0, a.c1), B::add_raw(b.c0, b.c1)), B::p2x2());
    Wide t = B::mul_wide(a.c0, b.c0);
    Wide re = B::add_wide(t, B::p2x2());
    im = B::sub_wide(im, t);
    t = B::mul_wide(a.c1, b.c1);
    re = B::sub_wide(re, t);
    im = B::sub_wide(im, t);
    t = B::mul_wide(c.c1, d.c1);
    re = B::add_wide(re, t);
    im = B::add_wide(im, t);
    t = B::mul_wide(c.c0, d.c0);
    re = B::sub_wide(re, t);
    im = B::add_wide(im, t);
    im = B::sub_wide(im, B::mul_wide(B::add_raw(c.c0, c.c1), B::add_raw(d.c0, d.c1)));
    return Fp2{B::redc(re), B::redc(im)};
  }
  ZKB_HD static Fp2 mul(const Fp2& a, const Fp2& b) { return mul_v(a, b); }
  ZKB_HD static Fp2 sqr(const Fp2& a) { return sqr_v(a); }
  ZKB_HD static Fp2 mul_sub(const Fp2& a, const Fp2& b, const Fp2& c, const Fp2& d) { return mul_sub_v(a, b, c, d); }
  ZKB_HD static Fp2 mul_ni(const Fp2& a, const Fp2& b) { return mul_v(a, b); }
  ZKB_NI static Fp2 inv(const Fp2& a) {
    B d = B::inv(B::add(B::sqr(a.c0), B::sqr(a.c1)));
    return Fp2{B::mul(a.c0, d), B::neg(B::mul(a.c1, d))};
  }
  ZKB_HD static Fp2 to_mont(const Fp2& a) { return Fp2{B::to_mont(a.c0), B::to_mont(a.c1)}; }
  ZKB_HD static Fp2 from_mont(const Fp2& a) { return Fp2{B::from_mont(a.c0), B::from_mont(a.c1)}; }
};

template <class P>
using Fp2 = Fp2T<Fp<P>>;

}  // namespace zkb
