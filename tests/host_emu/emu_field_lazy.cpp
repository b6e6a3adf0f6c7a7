// Host emulation harness (TEST ONLY) for the lazy-reduction arithmetic: fp.cuh, fp2.cuh and ec.cuh compiled as plain
// C++ (-DZKB_EMU).  Every entry point runs one operation over `n` cases laid out back to back as 32-bit limbs.
#include <string.h>

#include "ec.cuh"
using namespace zkb;

template <class T> static T take(const uint32_t*& p) {
  T r;
  memcpy(&r, p, sizeof(T));
  p += sizeof(T) / 4;
  return r;
}
template <class T> static void put(uint32_t*& p, const T& v) {
  memcpy(p, &v, sizeof(T));
  p += sizeof(T) / 4;
}

// op 0: sqr(a)  1: mul_sub(a, b, c, d)  2: mul_wide(a, b)  3: sqr_wide(a)  4: redc(T)
template <class P> static void fp_op(int op, const uint32_t* in, uint32_t* out, int n) {
  typedef Fp<P> F;
  for (int k = 0; k < n; k++) {
    if (op == 0) { F a = take<F>(in); put(out, F::sqr(a)); }
    if (op == 1) { F a = take<F>(in), b = take<F>(in), c = take<F>(in), d = take<F>(in); put(out, F::mul_sub(a, b, c, d)); }
    if (op == 2) { F a = take<F>(in), b = take<F>(in); put(out, F::mul_wide(a, b)); }
    if (op == 3) { F a = take<F>(in); put(out, F::sqr_wide(a)); }
    if (op == 4) { typename F::Wide t = take<typename F::Wide>(in); put(out, F::redc(t)); }
  }
}

// op 0: mul(a, b)  1: sqr(a)  2: mul_sub(a, b, c, d)
template <class P> static void fp2_op(int op, const uint32_t* in, uint32_t* out, int n) {
  typedef Fp2<P> F;
  for (int k = 0; k < n; k++) {
    if (op == 0) { F a = take<F>(in), b = take<F>(in); put(out, F::mul(a, b)); }
    if (op == 1) { F a = take<F>(in); put(out, F::sqr(a)); }
    if (op == 2) { F a = take<F>(in), b = take<F>(in), c = take<F>(in), d = take<F>(in); put(out, F::mul_sub(a, b, c, d)); }
  }
}

// op 0: madd(XYZZ a, Affine q)  1: add(XYZZ a, XYZZ b)  2: dbl(XYZZ a)  3: mdbl(Affine q); the result is an XYZZ point
template <class F> static void ec_op(int op, const uint32_t* in, uint32_t* out, int n) {
  typedef XYZZ<F> X;
  for (int k = 0; k < n; k++) {
    if (op == 0) { X a = take<X>(in); Affine<F> q = take<Affine<F>>(in); put(out, X::madd(a, q)); }
    if (op == 1) { X a = take<X>(in), b = take<X>(in); put(out, X::add(a, b)); }
    if (op == 2) { X a = take<X>(in); put(out, X::dbl(a)); }
    if (op == 3) { Affine<F> q = take<Affine<F>>(in); put(out, X::mdbl(q)); }
  }
}

// field: 0 BN254 Fr, 1 BN254 Fq, 2 BLS12-381 Fr, 3 BLS12-381 Fq
extern "C" void emu_lazy_fp(int field, int op, const uint32_t* in, uint32_t* out, int n) {
  switch (field) {
    case 0: fp_op<Bn254Fr>(op, in, out, n); break;
    case 1: fp_op<Bn254Fq>(op, in, out, n); break;
    case 2: fp_op<Bls381Fr>(op, in, out, n); break;
    case 3: fp_op<Bls381Fq>(op, in, out, n); break;
  }
}

// curve: 0 BN254, 1 BLS12-381
extern "C" void emu_lazy_fp2(int curve, int op, const uint32_t* in, uint32_t* out, int n) {
  if (curve == 0) fp2_op<Bn254Fq>(op, in, out, n);
  else fp2_op<Bls381Fq>(op, in, out, n);
}

// group: 1 G1, 2 G2
extern "C" void emu_lazy_ec(int curve, int group, int op, const uint32_t* in, uint32_t* out, int n) {
  if (curve == 0) {
    if (group == 1) ec_op<Fp<Bn254Fq>>(op, in, out, n);
    else ec_op<Fp2<Bn254Fq>>(op, in, out, n);
  } else {
    if (group == 1) ec_op<Fp<Bls381Fq>>(op, in, out, n);
    else ec_op<Fp2<Bls381Fq>>(op, in, out, n);
  }
}
