// Host-side Montgomery arithmetic on 64-bit limbs with the same static interface as Fp<P>, used only
// for the serial tail of the prover (window Horner, five scalar multiplications, three affine
// conversions — row a3 of SURVEY.md §8: "final combination ... glue").  Measured on B200 a single GPU
// thread needs ~0.3 us per dependent 256-bit multiplication (8.3 ms for the whole tail); a host core
// needs ~30 ns, and ark performs the same tail on the CPU
// (ark-groth16 create_proof_with_reduction, reached from /root/reference/zokrates_ark/src/groth16.rs:44).
//
// Memory layout equals Fp<P> (little-endian limbs, same Montgomery radix R = 2^(32 P::N)), so device
// results are reinterpreted without conversion.
#pragma once
#include "fp.cuh"

namespace zkb {

template <class P>
struct alignas(16) Fp64 {
  static constexpr int N = P::N / 2;
  typedef P Params;
  typedef unsigned __int128 u128;
  uint64_t v[N];

  ZKB_HD static uint64_t modl(int i) { return ((uint64_t)P::mod(2 * i + 1) << 32) | P::mod(2 * i); }
  ZKB_HD static uint64_t inv64() {
    // P::INV = -p^-1 mod 2^32; lift p^-1 to 64 bits with one Newton step
    uint64_t p0 = modl(0);
    uint64_t x = (uint64_t)(uint32_t)(0u - P::INV);
    x = x * (2 - p0 * x);
    return (uint64_t)0 - x;
  }
  ZKB_HD static Fp64 zero() { Fp64 r; for (int i = 0; i < N; i++) r.v[i] = 0; return r; }
  ZKB_HD static Fp64 one() { Fp64 r; for (int i = 0; i < N; i++) r.v[i] = ((uint64_t)P::r1(2 * i + 1) << 32) | P::r1(2 * i); return r; }
  ZKB_HD static Fp64 r2() { Fp64 r; for (int i = 0; i < N; i++) r.v[i] = ((uint64_t)P::r2(2 * i + 1) << 32) | P::r2(2 * i); return r; }
  ZKB_HD bool is_zero() const { uint64_t a = 0; for (int i = 0; i < N; i++) a |= v[i]; return a == 0; }
  ZKB_HD bool operator==(const Fp64& o) const { uint64_t a = 0; for (int i = 0; i < N; i++) a |= v[i] ^ o.v[i]; return a == 0; }
  ZKB_HD bool operator!=(const Fp64& o) const { return !(*this == o); }
  ZKB_HD static bool geq_p(const Fp64& a) {
    for (int i = N - 1; i >= 0; i--) { uint64_t m = modl(i); if (a.v[i] > m) return true; if (a.v[i] < m) return false; }
    return true;
  }
  ZKB_HD static Fp64 sub_p(const Fp64& a) {
    Fp64 r; uint64_t borrow = 0;
    for (int i = 0; i < N; i++) { u128 d = (u128)a.v[i] - modl(i) - borrow; r.v[i] = (uint64_t)d; borrow = (uint64_t)(d >> 64) & 1; }
    return r;
  }
  ZKB_HD static Fp64 add(const Fp64& a, const Fp64& b) {
    Fp64 t; uint64_t c = 0;
    for (int i = 0; i < N; i++) { u128 s = (u128)a.v[i] + b.v[i] + c; t.v[i] = (uint64_t)s; c = (uint64_t)(s >> 64); }
    return (c || geq_p(t)) ? sub_p(t) : t;
  }
  ZKB_HD static Fp64 sub(const Fp64& a, const Fp64& b) {
    Fp64 t; uint64_t borrow = 0;
    for (int i = 0; i < N; i++) { u128 d = (u128)a.v[i] - b.v[i] - borrow; t.v[i] = (uint64_t)d; borrow = (uint64_t)(d >> 64) & 1; }
    if (borrow) { uint64_t c = 0; for (int i = 0; i < N; i++) { u128 s = (u128)t.v[i] + modl(i) + c; t.v[i] = (uint64_t)s; c = (uint64_t)(s >> 64); } }
    return t;
  }
  ZKB_HD static Fp64 neg(const Fp64& a) { return a.is_zero() ? a : sub(zero(), a); }
  ZKB_HD static Fp64 dbl(const Fp64& a) { return add(a, a); }
  ZKB_HD static Fp64 mul(const Fp64& a, const Fp64& b) {
    uint64_t t[N + 2];
    for (int i = 0; i < N + 2; i++) t[i] = 0;
    const uint64_t inv = inv64();
    for (int i = 0; i < N; i++) {
      uint64_t c = 0;
      for (int j = 0; j < N; j++) { u128 s = (u128)a.v[j] * b.v[i] + t[j] + c; t[j] = (uint64_t)s; c = (uint64_t)(s >> 64); }
      u128 s2 = (u128)t[N] + c; t[N] = (uint64_t)s2; t[N + 1] = (uint64_t)(s2 >> 64);
      uint64_t m = t[0] * inv;
      u128 s = (u128)m * modl(0) + t[0]; c = (uint64_t)(s >> 64);
      for (int j = 1; j < N; j++) { s = (u128)m * modl(j) + t[j] + c; t[j - 1] = (uint64_t)s; c = (uint64_t)(s >> 64); }
      s2 = (u128)t[N] + c; t[N - 1] = (uint64_t)s2; t[N] = t[N + 1] + (uint64_t)(s2 >> 64);
    }
    Fp64 o; for (int i = 0; i < N; i++) o.v[i] = t[i];
    return (t[N] || geq_p(o)) ? sub_p(o) : o;
  }
  ZKB_HD static Fp64 sqr(const Fp64& a) { return mul(a, a); }
  ZKB_HD static Fp64 mul_sub(const Fp64& a, const Fp64& b, const Fp64& c, const Fp64& d) { return sub(mul(a, b), mul(c, d)); }

  // the lazy-reduction interface of Fp<P> (used by Fp2T): unreduced 2N-limb products and one reduction per sum
  struct Wide {
    uint64_t v[2 * N];
  };
  ZKB_HD static Fp64 add_raw(const Fp64& a, const Fp64& b) {
    Fp64 t; uint64_t c = 0;
    for (int i = 0; i < N; i++) { u128 s = (u128)a.v[i] + b.v[i] + c; t.v[i] = (uint64_t)s; c = (uint64_t)(s >> 64); }
    return t;
  }
  ZKB_HD static Wide mul_wide(const Fp64& a, const Fp64& b) {
    Wide t;
    for (int i = 0; i < 2 * N; i++) t.v[i] = 0;
    for (int i = 0; i < N; i++) {
      uint64_t c = 0;
      for (int j = 0; j < N; j++) { u128 s = (u128)a.v[j] * b.v[i] + t.v[i + j] + c; t.v[i + j] = (uint64_t)s; c = (uint64_t)(s >> 64); }
      t.v[i + N] = c;
    }
    return t;
  }
  ZKB_HD static Wide sqr_wide(const Fp64& a) { return mul_wide(a, a); }
  ZKB_HD static Fp64 redc(const Wide& T) {  // T < p R
    uint64_t t[2 * N + 1];
    for (int i = 0; i < 2 * N; i++) t[i] = T.v[i];
    t[2 * N] = 0;
    const uint64_t inv = inv64();
    for (int i = 0; i < N; i++) {
      const uint64_t m = t[i] * inv;
      uint64_t c = 0;
      for (int j = 0; j < N; j++) { u128 s = (u128)m * modl(j) + t[i + j] + c; t[i + j] = (uint64_t)s; c = (uint64_t)(s >> 64); }
      for (int k = i + N; c && k <= 2 * N; k++) { u128 s = (u128)t[k] + c; t[k] = (uint64_t)s; c = (uint64_t)(s >> 64); }
    }
    Fp64 o; for (int i = 0; i < N; i++) o.v[i] = t[N + i];
    return (t[2 * N] || geq_p(o)) ? sub_p(o) : o;
  }
  ZKB_HD static Wide add_wide(const Wide& a, const Wide& b) {
    Wide t; uint64_t c = 0;
    for (int i = 0; i < 2 * N; i++) { u128 s = (u128)a.v[i] + b.v[i] + c; t.v[i] = (uint64_t)s; c = (uint64_t)(s >> 64); }
    return t;
  }
  ZKB_HD static Wide sub_wide(const Wide& a, const Wide& b) {
    Wide t; uint64_t borrow = 0;
    for (int i = 0; i < 2 * N; i++) { u128 d = (u128)a.v[i] - b.v[i] - borrow; t.v[i] = (uint64_t)d; borrow = (uint64_t)(d >> 64) & 1; }
    return t;
  }
  ZKB_HD static Wide p2() { Wide t; for (int i = 0; i < 2 * N; i++) t.v[i] = ((uint64_t)P::p2(2 * i + 1) << 32) | P::p2(2 * i); return t; }
  ZKB_HD static Wide p2x2() { Wide t; for (int i = 0; i < 2 * N; i++) t.v[i] = ((uint64_t)P::p2x2(2 * i + 1) << 32) | P::p2x2(2 * i); return t; }
  ZKB_HD static Fp64 mul_ni(const Fp64& a, const Fp64& b) { return mul(a, b); }
  ZKB_HD static Fp64 to_mont(const Fp64& a) { return mul(a, r2()); }
  ZKB_HD static Fp64 from_mont(const Fp64& a) { Fp64 o = zero(); o.v[0] = 1; return mul(a, o); }
  ZKB_HD static Fp64 inv(const Fp64& a) {
    // a^(p-2)
    uint64_t e[N];
    for (int i = 0; i < N; i++) e[i] = modl(i);
    uint64_t borrow = 2;
    for (int i = 0; i < N && borrow; i++) { uint64_t o = e[i]; e[i] = o - borrow; borrow = o < borrow ? 1 : 0; }
    Fp64 r = one();
    bool started = false;
    for (int i = N - 1; i >= 0; i--)
      for (int b = 63; b >= 0; b--) {
        if (started) r = mul(r, r);
        if ((e[i] >> b) & 1) { r = started ? mul(r, a) : a; started = true; }
      }
    return r;
  }
};

}  // namespace zkb
