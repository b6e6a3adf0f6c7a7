// Montgomery-form prime-field arithmetic on 32-bit limbs (8 limbs: BN254 Fr/Fq, BLS12-381 Fr;
// 12 limbs: BLS12-381 Fq).
//
// Replaces, on the device, what the reference reaches through `zokrates_field::FieldPrime`
// (/root/reference/zokrates_field/src/lib.rs:407-503 -> ark_ff::Fp256/Fp384 Montgomery ops, ark-ff
// 0.3.0, Cargo.lock:161).  Values are the same residues; the limb width (32 vs ark's 64) and the
// Montgomery radix R = 2^(32 N) = 2^256 / 2^384 coincide with ark's, so Montgomery images are
// bit-identical to ark's in-memory representation.
//
// mul(): CIOS Montgomery multiplication with the product columns split into an "even" and an
// "odd" accumulator so that every 32x32->64 product is ONE multiply-add (IMAD.WIDE.U32 with a
// predicate carry) and each row is two independent carry chains: N*(2N+1) wide MADs per
// multiplication (136 for N = 8, 300 for N = 12) — the unit SURVEY.md §8(d) counts.
//
// Lazy reduction for the curve formulas: mul_wide / sqr_wide return the 2N-limb product without a
// reduction and redc() reduces it, so sums and differences of products pay for ONE reduction:
// mul_wide N^2 wide MADs, sqr_wide N(N+1)/2 (cross products once, doubled, then the diagonal), redc N^2 + N.
// Bounds: redc needs its input < p R, which takes 2p < R for mul_sub and the Fq2 c0 (inputs < 2p^2),
// and 4p < R for fp2.cuh mul_sub_v (inputs < 4p^2).
//   BN254:          p < 2^254, R = 2^256.
//   BLS12-381 Fq:   p < 2^381, R = 2^384.
// Both fields satisfy both conditions; static_asserts on P::BITS stop the build for a field that does not.
#pragma once
#include "hd.cuh"
#include "field_params.cuh"

namespace zkb {

template <class P>
struct alignas(16) Fp {
  static constexpr int N = P::N;
  typedef P Params;
  uint32_t v[N];

  ZKB_HD static Fp zero() {
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = 0;
    return r;
  }
  ZKB_HD static Fp one() {  // Montgomery image of 1
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = P::r1(i);
    return r;
  }
  ZKB_HD static Fp r2() {
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = P::r2(i);
    return r;
  }
  ZKB_HD static Fp modulus() {
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = P::mod(i);
    return r;
  }
  ZKB_HD bool is_zero() const {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < N; i++) acc |= v[i];
    return acc == 0;
  }
  ZKB_HD bool operator==(const Fp& o) const {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < N; i++) acc |= v[i] ^ o.v[i];
    return acc == 0;
  }
  ZKB_HD bool operator!=(const Fp& o) const { return !(*this == o); }

  // r = a - p if a >= p else a   (a < 2p)
  ZKB_HD static Fp reduce_once(const Fp& a) {
    Fp t;
    t.v[0] = ptx::sub_cc(a.v[0], P::mod(0));
#pragma unroll
    for (int i = 1; i < N; i++) t.v[i] = ptx::subc_cc(a.v[i], P::mod(i));
    uint32_t borrow = ptx::subc(0, 0);  // 0 - 0 - CF  -> 0xffffffff when a < p
    Fp r;
#pragma unroll
    for (int i = 0; i < N; i++) r.v[i] = borrow ? a.v[i] : t.v[i];
    return r;
  }

  ZKB_HD static Fp add(const Fp& a, const Fp& b) {
    Fp t;  // 2p < 2^(32N) for every field here, so the raw sum does not overflow
    t.v[0] = ptx::add_cc(a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t.v[i] = ptx::addc_cc(a.v[i], b.v[i]);
    t.v[N - 1] = ptx::addc(a.v[N - 1], b.v[N - 1]);
    return reduce_once(t);
  }

  ZKB_HD static Fp sub(const Fp& a, const Fp& b) {
    Fp t;
    t.v[0] = ptx::sub_cc(a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < N; i++) t.v[i] = ptx::subc_cc(a.v[i], b.v[i]);
    uint32_t borrow = ptx::subc(0, 0);  // all-ones when a < b
    Fp r;
    r.v[0] = ptx::add_cc(t.v[0], P::mod(0) & borrow);
#pragma unroll
    for (int i = 1; i < N - 1; i++) r.v[i] = ptx::addc_cc(t.v[i], P::mod(i) & borrow);
    r.v[N - 1] = ptx::addc(t.v[N - 1], P::mod(N - 1) & borrow);
    return r;
  }

  ZKB_HD static Fp neg(const Fp& a) {
    if (a.is_zero()) return a;
    Fp r;
    r.v[0] = ptx::sub_cc(P::mod(0), a.v[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) r.v[i] = ptx::subc_cc(P::mod(i), a.v[i]);
    r.v[N - 1] = ptx::subc(P::mod(N - 1), a.v[N - 1]);
    return r;
  }

  ZKB_HD static Fp dbl(const Fp& a) { return add(a, a); }

  // Rows of the product a * b on the even / odd accumulators: E[k] holds word k and O[k] word k + 1, so the words of
  // one row are two carry chains of one IMAD.WIDE.U32(.X) each.  First row: (E, O) = a * y.
  ZKB_HD static void row_first(uint32_t* E, uint32_t* O, const Fp& a, uint32_t y) {
#pragma unroll
    for (int j = 0; j < N; j += 2) {
      uint64_t w = (uint64_t)a.v[j] * y;
      E[j] = (uint32_t)w;
      E[j + 1] = (uint32_t)(w >> 32);
      uint64_t u = (uint64_t)a.v[j + 1] * y;
      O[j] = (uint32_t)u;
      O[j + 1] = (uint32_t)(u >> 32);
    }
  }
  // Next row: (E, O) <- (E, O) / W + a * y; word 0 of E has been consumed (cancelled or stored) by the caller.
  ZKB_HD static void row_next(uint32_t* E, uint32_t* O, const Fp& a, uint32_t y) {
    uint32_t nE[N], nO[N];
    nE[0] = ptx::add_cc(O[0], E[1]);
#pragma unroll
    for (int j = 1; j < N - 1; j += 2) ptx::madc_wide_cc(nO[j - 1], nO[j], a.v[j], y, E[j + 1], E[j + 2]);
    ptx::madc_wide(nO[N - 2], nO[N - 1], a.v[N - 1], y, 0, 0);
    ptx::mad_wide_cc(nE[0], nE[1], a.v[0], y, nE[0], O[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) ptx::madc_wide_cc(nE[j], nE[j + 1], a.v[j], y, O[j], O[j + 1]);
    nO[N - 1] = ptx::addc(nO[N - 1], 0);
#pragma unroll
    for (int j = 0; j < N; j++) {
      E[j] = nE[j];
      O[j] = nO[j];
    }
  }

  // Montgomery product a*b*R^-1 mod p, fully reduced.
  ZKB_HD static Fp mul(const Fp& a, const Fp& b) {
    static_assert(N % 2 == 0, "even limb count");
    // T = sum E[k] W^k + sum O[k] W^(k+1)
    uint32_t E[N], O[N];
    row_first(E, O, a, b.v[0]);
#pragma unroll
    for (int i = 0; i < N; i++) {
      // shift one word down (E[0] == 0 after the previous reduction) and add a * b[i]
      if (i > 0) row_next(E, O, a, b.v[i]);
      // T += m * p with m chosen so that word 0 cancels
      const uint32_t m = E[0] * P::INV;
      ptx::mad_wide_cc(O[0], O[1], P::mod(1), m, O[0], O[1]);
#pragma unroll
      for (int j = 3; j < N; j += 2) ptx::madc_wide_cc(O[j - 1], O[j], P::mod(j), m, O[j - 1], O[j]);
      ptx::mad_wide_cc(E[0], E[1], P::mod(0), m, E[0], E[1]);
#pragma unroll
      for (int j = 2; j < N; j += 2) ptx::madc_wide_cc(E[j], E[j + 1], P::mod(j), m, E[j], E[j + 1]);
      O[N - 1] = ptx::addc(O[N - 1], 0);
    }
    // result = T / W = O + (E >> 32)
    Fp t;
    t.v[0] = ptx::add_cc(O[0], E[1]);
#pragma unroll
    for (int k = 1; k < N - 1; k++) t.v[k] = ptx::addc_cc(O[k], E[k + 1]);
    t.v[N - 1] = ptx::addc(O[N - 1], 0);
    return reduce_once(t);
  }

  // ---- lazy reduction -------------------------------------------------------------------------------------------
  struct Wide {  // 2N-limb unreduced value, little-endian
    uint32_t v[2 * N];
  };

  // a + b without the final subtraction: < 2p, the operand of a product whose sum is reduced later
  ZKB_HD static Fp add_raw(const Fp& a, const Fp& b) {
    Fp t;
    t.v[0] = ptx::add_cc(a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t.v[i] = ptx::addc_cc(a.v[i], b.v[i]);
    t.v[N - 1] = ptx::addc(a.v[N - 1], b.v[N - 1]);
    return t;
  }

  // a * b on 2N limbs (a, b < 2^(32N)): N^2 wide MADs, the rows of mul() without the reduction
  ZKB_HD static Wide mul_wide(const Fp& a, const Fp& b) {
    Wide t;
    uint32_t E[N], O[N];
    row_first(E, O, a, b.v[0]);
    t.v[0] = E[0];
#pragma unroll
    for (int i = 1; i < N; i++) {
      row_next(E, O, a, b.v[i]);
      t.v[i] = E[0];  // word i is final: later rows start at word i + 1
    }
    t.v[N] = ptx::add_cc(O[0], E[1]);
#pragma unroll
    for (int k = 1; k < N - 1; k++) t.v[N + k] = ptx::addc_cc(O[k], E[k + 1]);
    t.v[2 * N - 1] = ptx::addc(O[N - 1], 0);
    return t;
  }

  // Cross products of sqr_wide, row i <= N - 2: z += a_i * a_j W^(i + j) for j = j0, j0 + 2, ... < N.  The pairs of one
  // row do not overlap, so they are one carry chain; it runs on to word i + N, the highest one that rows before i may have
  // set, and ends in word i + N + 1, which is still zero.  (Constant loop bounds: every copy unrolls.)
  ZKB_HD static void cross_row(uint32_t* z, const Fp& a, int i, int j0) {
    if (j0 >= N) return;
#pragma unroll
    for (int j = 1; j < N; j++) {
      if (j < j0 || ((j - j0) & 1)) continue;
      if (j == j0) ptx::mad_wide_cc(z[i + j], z[i + j + 1], a.v[j], a.v[i], z[i + j], z[i + j + 1]);
      else ptx::madc_wide_cc(z[i + j], z[i + j + 1], a.v[j], a.v[i], z[i + j], z[i + j + 1]);
    }
    if ((N - 1 - j0) & 1) z[i + N] = ptx::addc_cc(z[i + N], 0);  // the last pair ended at word i + N - 1
    z[i + N + 1] = ptx::addc(z[i + N + 1], 0);
  }

  // a^2 on 2N limbs: the N(N-1)/2 cross products once (words of even / odd position in two accumulators, so that no two
  // products of one chain overlap), doubled by a one-bit shift, plus the N squares on the diagonal: N(N+1)/2 wide MADs
  ZKB_HD static Wide sqr_wide(const Fp& a) {
    uint32_t X[2 * N], Y[2 * N];
#pragma unroll
    for (int k = 0; k < 2 * N; k++) X[k] = Y[k] = 0;
#pragma unroll
    for (int i = 0; i < N - 1; i++) {
      cross_row(X, a, i, i + 1);  // i + j odd
      cross_row(Y, a, i, i + 2);  // i + j even
    }
    Wide t;
    t.v[0] = ptx::add_cc(X[0], Y[0]);
#pragma unroll
    for (int k = 1; k < 2 * N - 1; k++) t.v[k] = ptx::addc_cc(X[k], Y[k]);
    t.v[2 * N - 1] = ptx::addc(X[2 * N - 1], Y[2 * N - 1]);
#pragma unroll
    for (int k = 2 * N - 1; k > 0; k--) t.v[k] = (t.v[k] << 1) | (t.v[k - 1] >> 31);
    t.v[0] <<= 1;
    ptx::mad_wide_cc(t.v[0], t.v[1], a.v[0], a.v[0], t.v[0], t.v[1]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) ptx::madc_wide_cc(t.v[2 * i], t.v[2 * i + 1], a.v[i], a.v[i], t.v[2 * i], t.v[2 * i + 1]);
    ptx::madc_wide(t.v[2 * N - 2], t.v[2 * N - 1], a.v[N - 1], a.v[N - 1], t.v[2 * N - 2], t.v[2 * N - 1]);
    return t;
  }

  // Montgomery reduction T*R^-1 mod p of T < p*R, fully reduced: N^2 + N wide MADs.  Row i cancels word i with
  // m = word * (-p^-1) and adds word N + i - 1 of T at the top of the (E, O) window; every intermediate is
  // < R + (W + 1) p, which fits the window when 2p < R.
  ZKB_HD static Fp redc(const Wide& T) {
    static_assert(P::BITS + 1 <= 32 * N, "redc needs 2p < R");
    uint32_t E[N], O[N];
    {
      const uint32_t m = T.v[0] * P::INV;
#pragma unroll
      for (int j = 1; j < N; j += 2) {
        uint64_t u = (uint64_t)P::mod(j) * m;
        O[j - 1] = (uint32_t)u;
        O[j] = (uint32_t)(u >> 32);
      }
      ptx::mad_wide_cc(E[0], E[1], P::mod(0), m, T.v[0], T.v[1]);
#pragma unroll
      for (int j = 2; j < N; j += 2) ptx::madc_wide_cc(E[j], E[j + 1], P::mod(j), m, T.v[j], T.v[j + 1]);
      O[N - 1] = ptx::addc(O[N - 1], 0);
    }
#pragma unroll
    for (int i = 1; i < N; i++) {
      // the row_next() shift with m * p as the row; m needs word 0 of the shifted window, so it is computed between
      // the add that forms that word and the chain that takes its carry (a plain multiply leaves the carry flag alone)
      uint32_t nE[N], nO[N];
      nE[0] = ptx::add_cc(O[0], E[1]);
      const uint32_t m = nE[0] * P::INV;
#pragma unroll
      for (int j = 1; j < N - 1; j += 2) ptx::madc_wide_cc(nO[j - 1], nO[j], P::mod(j), m, E[j + 1], E[j + 2]);
      ptx::madc_wide(nO[N - 2], nO[N - 1], P::mod(N - 1), m, T.v[N + i - 1], 0);
      ptx::mad_wide_cc(nE[0], nE[1], P::mod(0), m, nE[0], O[1]);
#pragma unroll
      for (int j = 2; j < N; j += 2) ptx::madc_wide_cc(nE[j], nE[j + 1], P::mod(j), m, O[j], O[j + 1]);
      nO[N - 1] = ptx::addc(nO[N - 1], 0);
#pragma unroll
      for (int j = 0; j < N; j++) {
        E[j] = nE[j];
        O[j] = nO[j];
      }
    }
    // (T + m p) / R = O + (E >> 32) + T[2N-1] W^(N-1) < 2p
    Fp t;
    t.v[0] = ptx::add_cc(O[0], E[1]);
#pragma unroll
    for (int k = 1; k < N - 1; k++) t.v[k] = ptx::addc_cc(O[k], E[k + 1]);
    t.v[N - 1] = ptx::addc(O[N - 1], T.v[2 * N - 1]);
    return reduce_once(t);
  }

  ZKB_HD static Wide add_wide(const Wide& a, const Wide& b) {
    Wide t;
    t.v[0] = ptx::add_cc(a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < 2 * N - 1; i++) t.v[i] = ptx::addc_cc(a.v[i], b.v[i]);
    t.v[2 * N - 1] = ptx::addc(a.v[2 * N - 1], b.v[2 * N - 1]);
    return t;
  }
  // a - b for a >= b
  ZKB_HD static Wide sub_wide(const Wide& a, const Wide& b) {
    Wide t;
    t.v[0] = ptx::sub_cc(a.v[0], b.v[0]);
#pragma unroll
    for (int i = 1; i < 2 * N - 1; i++) t.v[i] = ptx::subc_cc(a.v[i], b.v[i]);
    t.v[2 * N - 1] = ptx::subc(a.v[2 * N - 1], b.v[2 * N - 1]);
    return t;
  }
  ZKB_HD static Wide p2() {  // p^2
    Wide t;
#pragma unroll
    for (int i = 0; i < 2 * N; i++) t.v[i] = P::p2(i);
    return t;
  }
  ZKB_HD static Wide p2x2() {  // 2 p^2
    Wide t;
#pragma unroll
    for (int i = 0; i < 2 * N; i++) t.v[i] = P::p2x2(i);
    return t;
  }

  ZKB_HD static Fp sqr(const Fp& a) { return redc(sqr_wide(a)); }
  // a*b - c*d: redc(a b + p^2 - c d), an input in (0, 2p^2) < p R
  ZKB_HD static Fp mul_sub(const Fp& a, const Fp& b, const Fp& c, const Fp& d) {
    return redc(sub_wide(add_wide(mul_wide(a, b), p2()), mul_wide(c, d)));
  }
  // out-of-line copies for cold code (scalar multiplications, inversions, final combination): keeps
  // code size and compile time down; hot kernels use the inlined mul().
  ZKB_NI static Fp mul_ni(const Fp& a, const Fp& b) { return mul(a, b); }

  ZKB_HD static Fp to_mont(const Fp& a) { return mul(a, r2()); }
  ZKB_HD static Fp from_mont(const Fp& a) {
    Fp o = zero();
    o.v[0] = 1;
    return mul(a, o);
  }

  // a^e for a little-endian 32-bit-limb exponent with N limbs (square-and-multiply, MSB first)
  ZKB_NI static Fp pow_limbs(const Fp& a, const uint32_t* e, int nlimbs) {
    Fp r = one();
    bool started = false;
    for (int i = nlimbs - 1; i >= 0; i--) {
      for (int b = 31; b >= 0; b--) {
        if (started) r = mul_ni(r, r);
        if ((e[i] >> b) & 1) {
          r = started ? mul_ni(r, a) : a;
          started = true;
        }
      }
    }
    return r;
  }

  // Fermat inverse a^(p-2); inv(0) = 0
  ZKB_NI static Fp inv(const Fp& a) {
    uint32_t e[N];
#pragma unroll
    for (int i = 0; i < N; i++) e[i] = P::pm2(i);
    return pow_limbs(a, e, N);
  }

  ZKB_NI static Fp pow_u64(const Fp& a, uint64_t k) {
    uint32_t e[2] = {(uint32_t)k, (uint32_t)(k >> 32)};
    return pow_limbs(a, e, 2);
  }
};

}  // namespace zkb
