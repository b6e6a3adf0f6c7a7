// Short-Weierstrass group arithmetic (a = 0) generic over the coordinate field F (Fp<P> for G1,
// Fp2<P> for G2).  Replaces ark-ec 0.3.0 `GroupAffine`/`GroupProjective` add/double on the MSM
// path (external crate, Cargo.lock:146; reached from /root/reference/zokrates_ark/src/groth16.rs:44).
//
// Accumulators use extended Jacobian "XYZZ" coordinates (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2):
// mixed addition 8M + 2S (= 10 field multiplications, the SURVEY.md §8d accounting unit), full
// addition 12M + 2S, doubling 6M + 3S.  Results are representation independent: the affine point
// is canonical, so outputs are bit-identical to any other correct implementation.
//
// Y3 = R (Q - X3) - Y PPP is one F::mul_sub: both products unreduced, one Montgomery reduction.  The
// Pd / Rd zero tests below are exact only because every field operation returns the canonical
// residue (< p), never a merely congruent value.
#pragma once
#include "fp2.cuh"

namespace zkb {

template <class F>
struct Affine {
  F x, y;  // (0,0) encodes the point at infinity ((0,0) is never on y^2 = x^3 + b, b != 0)
  ZKB_HD bool is_inf() const { return x.is_zero() && y.is_zero(); }
  ZKB_HD static Affine inf() { return Affine{F::zero(), F::zero()}; }
  ZKB_HD static Affine neg(const Affine& p) { return Affine{p.x, F::neg(p.y)}; }
};

template <class F>
struct XYZZ {
  F x, y, zz, zzz;

  ZKB_HD static XYZZ identity() { return XYZZ{F::zero(), F::zero(), F::zero(), F::zero()}; }
  ZKB_HD bool is_identity() const { return zz.is_zero(); }
  ZKB_HD static XYZZ from_affine(const Affine<F>& p) {
    if (p.is_inf()) return identity();
    return XYZZ{p.x, p.y, F::one(), F::one()};
  }
  ZKB_HD static XYZZ neg(const XYZZ& p) { return XYZZ{p.x, F::neg(p.y), p.zz, p.zzz}; }

  // 2 * (affine p), p != infinity
  ZKB_HD static XYZZ mdbl(const Affine<F>& p) {
    F U = F::dbl(p.y);
    F V = F::sqr(U);
    F W = F::mul(U, V);
    F S = F::mul(p.x, V);
    F X2 = F::sqr(p.x);
    F M = F::add(F::dbl(X2), X2);
    F X3 = F::sub(F::sqr(M), F::dbl(S));
    F Y3 = F::mul_sub(M, F::sub(S, X3), W, p.y);
    return XYZZ{X3, Y3, V, W};
  }

  ZKB_HD static XYZZ dbl(const XYZZ& p) {
    F U = F::dbl(p.y);
    F V = F::sqr(U);
    F W = F::mul(U, V);
    F S = F::mul(p.x, V);
    F X2 = F::sqr(p.x);
    F M = F::add(F::dbl(X2), X2);
    F X3 = F::sub(F::sqr(M), F::dbl(S));
    F Y3 = F::mul_sub(M, F::sub(S, X3), W, p.y);
    return XYZZ{X3, Y3, F::mul(V, p.zz), F::mul(W, p.zzz)};  // identity stays identity (ZZ = 0)
  }

  // acc + (affine q): 8M + 2S on the generic path
  ZKB_HD static XYZZ madd(const XYZZ& a, const Affine<F>& q) {
    if (q.is_inf()) return a;
    if (a.is_identity()) return XYZZ{q.x, q.y, F::one(), F::one()};
    F U2 = F::mul(q.x, a.zz);
    F S2 = F::mul(q.y, a.zzz);
    F Pd = F::sub(U2, a.x);
    F Rd = F::sub(S2, a.y);
    if (Pd.is_zero()) {
      if (Rd.is_zero()) return mdbl_ni(q);
      return identity();
    }
    F PP = F::sqr(Pd);
    F PPP = F::mul(Pd, PP);
    F Q = F::mul(a.x, PP);
    F X3 = F::sub(F::sub(F::sqr(Rd), PPP), F::dbl(Q));
    F Y3 = F::mul_sub(Rd, F::sub(Q, X3), a.y, PPP);
    return XYZZ{X3, Y3, F::mul(a.zz, PP), F::mul(a.zzz, PPP)};
  }

  // a + b: 12M + 2S
  ZKB_HD static XYZZ add(const XYZZ& a, const XYZZ& b) {
    if (b.is_identity()) return a;
    if (a.is_identity()) return b;
    F U1 = F::mul(a.x, b.zz);
    F U2 = F::mul(b.x, a.zz);
    F S1 = F::mul(a.y, b.zzz);
    F S2 = F::mul(b.y, a.zzz);
    F Pd = F::sub(U2, U1);
    F Rd = F::sub(S2, S1);
    if (Pd.is_zero()) {
      if (Rd.is_zero()) return dbl_ni(a);
      return identity();
    }
    F PP = F::sqr(Pd);
    F PPP = F::mul(Pd, PP);
    F Q = F::mul(U1, PP);
    F X3 = F::sub(F::sub(F::sqr(Rd), PPP), F::dbl(Q));
    F Y3 = F::mul_sub(Rd, F::sub(Q, X3), S1, PPP);
    return XYZZ{X3, Y3, F::mul(F::mul(a.zz, b.zz), PP), F::mul(F::mul(a.zzz, b.zzz), PPP)};
  }

  // out-of-line copies for cold code
  ZKB_NI static XYZZ mdbl_ni(const Affine<F>& p) { return mdbl(p); }
  ZKB_NI static XYZZ dbl_ni(const XYZZ& p) { return dbl(p); }
  ZKB_NI static XYZZ add_ni(const XYZZ& a, const XYZZ& b) { return add(a, b); }
  ZKB_NI static XYZZ madd_ni(const XYZZ& a, const Affine<F>& q) { return madd(a, q); }

  ZKB_NI static Affine<F> to_affine(const XYZZ& p) {
    if (p.is_identity()) return Affine<F>::inf();
    F t = F::inv(F::mul(p.zz, p.zzz));
    F zzi = F::mul(t, p.zzz);
    F zzzi = F::mul(t, p.zz);
    return Affine<F>{F::mul(p.x, zzi), F::mul(p.y, zzzi)};
  }

  // k * base for a canonical (non-Montgomery) little-endian scalar of `nlimbs` 32-bit limbs
  ZKB_NI static XYZZ mul_affine(const Affine<F>& base, const uint32_t* k, int nlimbs) {
    XYZZ r = identity();
    for (int i = nlimbs - 1; i >= 0; i--)
      for (int b = 31; b >= 0; b--) {
        r = dbl_ni(r);
        if ((k[i] >> b) & 1) r = madd_ni(r, base);
      }
    return r;
  }
  ZKB_NI static XYZZ mul_xyzz(const XYZZ& base, const uint32_t* k, int nlimbs) {
    XYZZ r = identity();
    for (int i = nlimbs - 1; i >= 0; i--)
      for (int b = 31; b >= 0; b--) {
        r = dbl_ni(r);
        if ((k[i] >> b) & 1) r = add_ni(r, base);
      }
    return r;
  }
};

}  // namespace zkb
