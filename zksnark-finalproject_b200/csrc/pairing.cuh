// BLS12-381 pairing and Groth16 verification, one proof per thread (row f4 on the device).
//
// The device counterpart of host_pairing.hpp, over the Fq / Fq2 of mont.cuh / ec.cuh (lazy values in [0, 2q)).
// Everything is B2Z_HD, so the same code runs on the host through ptx.cuh's carry emulation (hostcheck.cu:
// b2z_host_verify_one, b2z_host_pairing_op) and is checked there against host_pairing.hpp.
//
//   tower      Fq6 = Fq2[v]/(v^3 - (1 + u)), Fq12 = Fq6[w]/(w^2 - v), as ark-ec models/bls12 (and host_pairing.hpp)
//   frobenius  a^q with the five constants gamma^k, gamma = (1 + u)^((q - 1) / 6), computed once on the host
//              (frobenius_consts) and handed to the kernels as a parameter
//   lines      M-type twist: B's line coefficients made on the fly by the homogeneous doubling / addition steps of
//              ark-ec's G2Prepared; gamma's and delta's come prepared in the pvk
//   final exp  easy part (q^6 - 1)(q^2 + 1), hard part by the x-power chain, exactly host_pairing.hpp's sequence;
//              squarings are the generic Fq12 squaring (no cyclotomic shortcut), so every intermediate value is the
//              same field element as on the host
//   decoding   zcash compressed points with arkworks' validation: flags, x < q, on the curve, and the r-order
//              subgroup decided by [r]P == O with the exact XYZZ group law of ec.cuh -- the host's own check, not an
//              endomorphism shortcut
#pragma once
#include "ec.cuh"
#include "inv_gcd.cuh"

namespace b2z {
namespace pairing {

// ------------------------------------------------------------------ Fq helpers
B2Z_HD FqEl fq_four() { return Fq::dbl(Fq::dbl(Fq::one())); }

// a > b for 12-limb integers
B2Z_HD bool limbs_gt(const uint32_t (&a)[12], const uint32_t (&b)[12]) {
  bool gt = false, decided = false;
#pragma unroll
  for (int i = 11; i >= 0; i--) {
    if (!decided && a[i] != b[i]) { gt = a[i] > b[i]; decided = true; }
  }
  return gt;
}

// canonical value > (q - 1) / 2  (arkworks' "lexicographically largest" for the sign flag)
B2Z_HD bool fq_is_larger(const FqEl& a) {
  constexpr uint32_t half[12] = {0xffffd555u, 0xdcff7fffu, 0x58a9ffffu, 0x0f55ffffu, 0x7b587b12u, 0xb3986950u,
                                 0x79c2895fu, 0xb23ba5c2u, 0x21a5d66bu, 0x258dd3dbu, 0x1cbff34du, 0x0d0088f5u};
  const FqEl c = Fq::from_mont(a);
  return limbs_gt(c.l, half);
}

// a / 2 (the Montgomery factor is unaffected): (a + (a odd ? q : 0)) >> 1 on the canonical representative
B2Z_HD FqEl fq_half(const FqEl& a) {
  const FqEl x = Fq::reduce(a);
  const uint32_t m = 0u - (x.l[0] & 1u);
  uint32_t t[12];
  uint64_t carry = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    const uint64_t s = (uint64_t)x.l[i] + (FqParams::p(i) & m) + carry;
    t[i] = (uint32_t)s;
    carry = s >> 32;
  }
  FqEl r;
#pragma unroll
  for (int i = 0; i < 11; i++) r.l[i] = (t[i] >> 1) | (t[i + 1] << 31);
  r.l[11] = (t[11] >> 1) | ((uint32_t)carry << 31);
  return r;
}

// q = 3 mod 4: sqrt(a) = a^((q + 1) / 4); false when a is a non-residue
B2Z_HD bool fq_sqrt(const FqEl& a, FqEl* out) {
  constexpr uint32_t e[12] = {0xffffeaabu, 0xee7fbfffu, 0xac54ffffu, 0x07aaffffu, 0x3dac3d89u, 0xd9cc34a8u,
                              0x3ce144afu, 0xd91dd2e1u, 0x90d2eb35u, 0x92c6e9edu, 0x8e5ff9a6u, 0x0680447au};
  uint32_t ev[12];
#pragma unroll
  for (int i = 0; i < 12; i++) ev[i] = e[i];
  const FqEl r = Fq::pow(a, ev, 12);
  *out = r;
  return Fq::eq(Fq::sqr(r), a);
}

// big-endian 48 bytes (first byte masked) -> Montgomery element; false when the integer is >= q
B2Z_HD bool fq_from_be(const uint8_t* s, uint8_t mask_first, FqEl* out) {
  FqEl c;
#pragma unroll
  for (int w = 0; w < 12; w++) {
    const int at = 44 - 4 * w;
    const uint32_t b0 = at == 0 ? (uint32_t)(s[0] & mask_first) : (uint32_t)s[at];
    c.l[w] = (b0 << 24) | ((uint32_t)s[at + 1] << 16) | ((uint32_t)s[at + 2] << 8) | (uint32_t)s[at + 3];
  }
  uint32_t q[12];
#pragma unroll
  for (int i = 0; i < 12; i++) q[i] = FqParams::p(i);
  if (!limbs_gt(q, c.l)) return false;
  *out = Fq::to_mont(c);
  return true;
}

// ------------------------------------------------------------------ Fq2 helpers
B2Z_HD Fq2El fq2_conj(const Fq2El& a) { return Fq2El{a.c0, Fq::neg(a.c1)}; }
B2Z_HD Fq2El fq2_mul_fq(const Fq2El& a, const FqEl& k) { return Fq2El{Fq::mul(a.c0, k), Fq::mul(a.c1, k)}; }
B2Z_HD Fq2El fq2_mul_xi(const Fq2El& a) { return Fq2El{Fq::sub(a.c0, a.c1), Fq::add(a.c0, a.c1)}; }   // * (1 + u)
B2Z_HD bool fq2_is_larger(const Fq2El& y) { return Fq::is_zero(y.c1) ? fq_is_larger(y.c0) : fq_is_larger(y.c1); }

// square root by the norm method (host_pairing.hpp's fq2_sqrt): any root, the caller picks the sign
inline B2Z_HD_NOINLINE bool fq2_sqrt(const Fq2El& a, Fq2El* out) {
  if (Fq2::is_zero(a)) { *out = a; return true; }
  FqEl s;
  if (Fq::is_zero(a.c1)) {
    if (fq_sqrt(a.c0, &s)) { *out = Fq2El{s, Fq::zero()}; return true; }
    if (fq_sqrt(Fq::neg(a.c0), &s)) { *out = Fq2El{Fq::zero(), s}; return true; }
    return false;
  }
  FqEl alpha, x0;
  if (!fq_sqrt(Fq::add(Fq::sqr(a.c0), Fq::sqr(a.c1)), &alpha)) return false;
  if (!fq_sqrt(fq_half(Fq::add(a.c0, alpha)), &x0))
    if (!fq_sqrt(fq_half(Fq::sub(a.c0, alpha)), &x0)) return false;
  const FqEl x1 = Fq::mul(a.c1, gcdinv::inv(Fq::dbl(x0)));
  *out = Fq2El{x0, x1};
  return Fq2::eq(Fq2::sqr(*out), a);
}

// ------------------------------------------------------------------ Fq6, Fq12
struct Fq6El {
  Fq2El c0, c1, c2;
};
struct Fq12El {
  Fq6El c0, c1;
};

B2Z_HD Fq6El fq6_zero() { return Fq6El{Fq2::zero(), Fq2::zero(), Fq2::zero()}; }
B2Z_HD Fq6El fq6_one() { return Fq6El{Fq2::one(), Fq2::zero(), Fq2::zero()}; }
B2Z_HD Fq6El fq6_add(const Fq6El& a, const Fq6El& b) { return Fq6El{Fq2::add(a.c0, b.c0), Fq2::add(a.c1, b.c1), Fq2::add(a.c2, b.c2)}; }
B2Z_HD Fq6El fq6_sub(const Fq6El& a, const Fq6El& b) { return Fq6El{Fq2::sub(a.c0, b.c0), Fq2::sub(a.c1, b.c1), Fq2::sub(a.c2, b.c2)}; }
B2Z_HD Fq6El fq6_neg(const Fq6El& a) { return Fq6El{Fq2::neg(a.c0), Fq2::neg(a.c1), Fq2::neg(a.c2)}; }
B2Z_HD Fq6El fq6_mul_v(const Fq6El& a) { return Fq6El{fq2_mul_xi(a.c2), a.c0, a.c1}; }   // * v  (v^3 = 1 + u)
B2Z_HD bool fq6_is_zero(const Fq6El& a) { return Fq2::is_zero(a.c0) && Fq2::is_zero(a.c1) && Fq2::is_zero(a.c2); }
B2Z_HD bool fq6_eq(const Fq6El& a, const Fq6El& b) { return Fq2::eq(a.c0, b.c0) && Fq2::eq(a.c1, b.c1) && Fq2::eq(a.c2, b.c2); }

// Karatsuba over Fq2: 6 Fq2 products
inline B2Z_HD_NOINLINE Fq6El fq6_mul(const Fq6El& a, const Fq6El& b) {
  const Fq2El t0 = Fq2::mul(a.c0, b.c0), t1 = Fq2::mul(a.c1, b.c1), t2 = Fq2::mul(a.c2, b.c2);
  const Fq2El x0 = Fq2::add(t0, fq2_mul_xi(Fq2::sub(Fq2::sub(Fq2::mul(Fq2::add(a.c1, a.c2), Fq2::add(b.c1, b.c2)), t1), t2)));
  const Fq2El x1 = Fq2::add(Fq2::sub(Fq2::sub(Fq2::mul(Fq2::add(a.c0, a.c1), Fq2::add(b.c0, b.c1)), t0), t1), fq2_mul_xi(t2));
  const Fq2El x2 = Fq2::add(Fq2::sub(Fq2::sub(Fq2::mul(Fq2::add(a.c0, a.c2), Fq2::add(b.c0, b.c2)), t0), t2), t1);
  return Fq6El{x0, x1, x2};
}
// a * (b0 + b1 v): 5 Fq2 products
inline B2Z_HD_NOINLINE Fq6El fq6_mul_by_01(const Fq6El& a, const Fq2El& b0, const Fq2El& b1) {
  const Fq2El t0 = Fq2::mul(a.c0, b0), t1 = Fq2::mul(a.c1, b1);
  const Fq2El x0 = Fq2::add(t0, fq2_mul_xi(Fq2::mul(a.c2, b1)));
  const Fq2El x1 = Fq2::sub(Fq2::sub(Fq2::mul(Fq2::add(a.c0, a.c1), Fq2::add(b0, b1)), t0), t1);
  const Fq2El x2 = Fq2::add(Fq2::mul(a.c2, b0), t1);
  return Fq6El{x0, x1, x2};
}
// a * (b1 v): 3 Fq2 products
B2Z_HD Fq6El fq6_mul_by_1(const Fq6El& a, const Fq2El& b1) {
  return Fq6El{fq2_mul_xi(Fq2::mul(a.c2, b1)), Fq2::mul(a.c0, b1), Fq2::mul(a.c1, b1)};
}
B2Z_HD Fq6El fq6_inv(const Fq6El& a) {
  const Fq2El t0 = Fq2::sub(Fq2::sqr(a.c0), fq2_mul_xi(Fq2::mul(a.c1, a.c2)));
  const Fq2El t1 = Fq2::sub(fq2_mul_xi(Fq2::sqr(a.c2)), Fq2::mul(a.c0, a.c1));
  const Fq2El t2 = Fq2::sub(Fq2::sqr(a.c1), Fq2::mul(a.c0, a.c2));
  const Fq2El d = Fq2::inv(Fq2::add(Fq2::mul(a.c0, t0), fq2_mul_xi(Fq2::add(Fq2::mul(a.c2, t1), Fq2::mul(a.c1, t2)))));
  return Fq6El{Fq2::mul(t0, d), Fq2::mul(t1, d), Fq2::mul(t2, d)};
}

B2Z_HD Fq12El fq12_one() { return Fq12El{fq6_one(), fq6_zero()}; }
B2Z_HD Fq12El fq12_conj(const Fq12El& a) { return Fq12El{a.c0, fq6_neg(a.c1)}; }   // = inverse on the cyclotomic subgroup
B2Z_HD bool fq12_is_zero(const Fq12El& a) { return fq6_is_zero(a.c0) && fq6_is_zero(a.c1); }
B2Z_HD bool fq12_eq(const Fq12El& a, const Fq12El& b) { return fq6_eq(a.c0, b.c0) && fq6_eq(a.c1, b.c1); }
B2Z_HD Fq12El fq12_reduce(const Fq12El& a) {
  Fq12El r = a;
  Fq2El* c = &r.c0.c0;
  for (int i = 0; i < 6; i++) c[i] = Fq2::reduce(c[i]);
  return r;
}

// Karatsuba: 3 Fq6 products
inline B2Z_HD_NOINLINE Fq12El fq12_mul(const Fq12El& a, const Fq12El& b) {
  const Fq6El t0 = fq6_mul(a.c0, b.c0), t1 = fq6_mul(a.c1, b.c1);
  const Fq6El m = fq6_mul(fq6_add(a.c0, a.c1), fq6_add(b.c0, b.c1));
  return Fq12El{fq6_add(t0, fq6_mul_v(t1)), fq6_sub(fq6_sub(m, t0), t1)};
}
// complex squaring: 2 Fq6 products.  (a0 + a1 w)^2 = (a0 + a1)(a0 + v a1) - t - v t  +  2 t w,  t = a0 a1
inline B2Z_HD_NOINLINE Fq12El fq12_sqr(const Fq12El& a) {
  const Fq6El t = fq6_mul(a.c0, a.c1);
  const Fq6El m = fq6_mul(fq6_add(a.c0, a.c1), fq6_add(a.c0, fq6_mul_v(a.c1)));
  return Fq12El{fq6_sub(fq6_sub(m, t), fq6_mul_v(t)), fq6_add(t, t)};
}
inline B2Z_HD_NOINLINE Fq12El fq12_inv(const Fq12El& a) {
  const Fq6El d = fq6_inv(fq6_sub(fq6_mul(a.c0, a.c0), fq6_mul_v(fq6_mul(a.c1, a.c1))));
  return Fq12El{fq6_mul(a.c0, d), fq6_neg(fq6_mul(a.c1, d))};
}
// f * (c0 + c1 v + c4 v w): the sparse line value of an M-type twist (ark-ec's Fp12::mul_by_014), 13 Fq2 products
inline B2Z_HD_NOINLINE Fq12El fq12_mul_by_014(const Fq12El& f, const Fq2El& c0, const Fq2El& c1, const Fq2El& c4) {
  const Fq6El aa = fq6_mul_by_01(f.c0, c0, c1);
  const Fq6El bb = fq6_mul_by_1(f.c1, c4);
  const Fq6El m = fq6_mul_by_01(fq6_add(f.c0, f.c1), c0, Fq2::add(c1, c4));
  return Fq12El{fq6_add(aa, fq6_mul_v(bb)), fq6_sub(fq6_sub(m, aa), bb)};
}

// gamma^1 .. gamma^5 for the Frobenius map, gamma = (1 + u)^((q - 1) / 6)
struct FrobConsts {
  Fq2El g[5];
};
inline FrobConsts frobenius_consts() {
  constexpr uint32_t e[12] = {0xfffff1c7u, 0x49aa7fffu, 0x72e35555u, 0x051caaaau, 0xd3c82906u, 0xe688231au,
                              0x7deb831fu, 0xe613e1ebu, 0xb5e1f223u, 0x0c849bf3u, 0x5eeaa66fu, 0x045582fcu};   // (q - 1) / 6
  const Fq2El base{Fq::one(), Fq::one()};
  Fq2El g = Fq2::one();
  for (int i = 12 * 32 - 1; i >= 0; i--) {
    g = Fq2::sqr(g);
    if ((e[i >> 5] >> (i & 31)) & 1) g = Fq2::mul(g, base);
  }
  FrobConsts fc;
  fc.g[0] = Fq2::reduce(g);
  for (int k = 1; k < 5; k++) fc.g[k] = Fq2::reduce(Fq2::mul(fc.g[k - 1], g));
  return fc;
}
// a^q
inline B2Z_HD_NOINLINE Fq12El fq12_frobenius(const Fq12El& a, const FrobConsts& fc) {
  Fq12El r;
  r.c0.c0 = fq2_conj(a.c0.c0);
  r.c0.c1 = Fq2::mul(fq2_conj(a.c0.c1), fc.g[1]);
  r.c0.c2 = Fq2::mul(fq2_conj(a.c0.c2), fc.g[3]);
  r.c1.c0 = Fq2::mul(fq2_conj(a.c1.c0), fc.g[0]);
  r.c1.c1 = Fq2::mul(fq2_conj(a.c1.c1), fc.g[2]);
  r.c1.c2 = Fq2::mul(fq2_conj(a.c1.c2), fc.g[4]);
  return r;
}

constexpr uint64_t kBlsX = 0xd201000000010000ull;   // |x|; x is negative

inline B2Z_HD_NOINLINE Fq12El fq12_exp_by_x(const Fq12El& a) {   // a^x for a in the cyclotomic subgroup
  Fq12El r = a;                                         // the leading bit of |x|
  for (int i = 62; i >= 0; i--) {
    r = fq12_sqr(r);
    if ((kBlsX >> i) & 1) r = fq12_mul(r, a);
  }
  return fq12_conj(r);
}

// ark-ec Bls12::final_exponentiation (host_pairing.hpp's sequence); false for f = 0
B2Z_HD bool final_exponentiation(const Fq12El& f, const FrobConsts& fc, Fq12El* out) {
  if (fq12_is_zero(f)) return false;
  Fq12El r = fq12_mul(fq12_conj(f), fq12_inv(f));
  r = fq12_mul(fq12_frobenius(fq12_frobenius(r, fc), fc), r);
  Fq12El y0 = fq12_sqr(r);
  Fq12El y1 = fq12_exp_by_x(r);
  Fq12El y2 = fq12_conj(r);
  y1 = fq12_mul(y1, y2);
  y2 = fq12_exp_by_x(y1);
  y1 = fq12_conj(y1);
  y1 = fq12_mul(y1, y2);
  y2 = fq12_exp_by_x(y1);
  y1 = fq12_frobenius(y1, fc);
  y1 = fq12_mul(y1, y2);
  r = fq12_mul(r, y0);
  y0 = fq12_exp_by_x(y1);
  y2 = fq12_exp_by_x(y0);
  y0 = fq12_frobenius(fq12_frobenius(y1, fc), fc);
  y1 = fq12_conj(y1);
  y1 = fq12_mul(y1, y2);
  y1 = fq12_mul(y1, y0);
  *out = fq12_mul(r, y1);
  return true;
}

// ------------------------------------------------------------------ decompression (zcash format, arkworks' checks)
B2Z_HD bool g1_in_subgroup(const AffinePoint<Fq>& p) {   // [r]P == O
  uint32_t r[8];
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = FrParams::p(i);
  return G1::is_identity(G1::mul_scalar(G1::from_affine(p), r));
}
B2Z_HD bool g2_in_subgroup(const AffinePoint<Fq2>& p) {
  uint32_t r[8];
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = FrParams::p(i);
  return G2::is_identity(G2::mul_scalar(G2::from_affine(p), r));
}

// false = malformed (host_pairing.hpp's g1_deserialize returns false): flags, x >= q, no square root, subgroup
inline B2Z_HD_NOINLINE bool g1_decompress(const uint8_t* s, AffinePoint<Fq>* out, bool* inf) {
  const uint8_t flags = s[0];
  *out = AffinePoint<Fq>{Fq::zero(), Fq::zero()};
  *inf = false;
  if (!(flags & 0x80)) return false;
  if (flags & 0x40) {
    if (flags & 0x3f) return false;
    for (int i = 1; i < 48; i++) if (s[i]) return false;
    *inf = true;
    return true;
  }
  FqEl x, y;
  if (!fq_from_be(s, 0x1f, &x)) return false;
  if (!fq_sqrt(Fq::add(Fq::mul(Fq::sqr(x), x), fq_four()), &y)) return false;
  if (fq_is_larger(y) != ((flags & 0x20) != 0)) y = Fq::neg(y);
  *out = AffinePoint<Fq>{x, Fq::reduce(y)};
  return g1_in_subgroup(*out);
}
inline B2Z_HD_NOINLINE bool g2_decompress(const uint8_t* s, AffinePoint<Fq2>* out, bool* inf) {
  const uint8_t flags = s[0];
  *out = AffinePoint<Fq2>{Fq2::zero(), Fq2::zero()};
  *inf = false;
  if (!(flags & 0x80)) return false;
  if (flags & 0x40) {
    if (flags & 0x3f) return false;
    for (int i = 1; i < 96; i++) if (s[i]) return false;
    *inf = true;
    return true;
  }
  Fq2El x, y;
  if (!fq_from_be(s, 0x1f, &x.c1) || !fq_from_be(s + 48, 0xff, &x.c0)) return false;
  const FqEl four = fq_four();
  if (!fq2_sqrt(Fq2::add(Fq2::mul(Fq2::sqr(x), x), Fq2El{four, four}), &y)) return false;
  if (fq2_is_larger(y) != ((flags & 0x20) != 0)) y = Fq2::neg(y);
  *out = AffinePoint<Fq2>{x, Fq2::reduce(y)};
  return g2_in_subgroup(*out);
}

// ------------------------------------------------------------------ G2 lines (ark-ec models/bls12/g2.rs, M-type)
struct LineCoeffs {
  Fq2El c0, c1, c2;
};
struct G2Homog {
  Fq2El x, y, z;
};
inline B2Z_HD_NOINLINE LineCoeffs line_double(G2Homog* r) {
  const FqEl two_inv = fq_half(Fq::one());
  const FqEl four = fq_four();
  const Fq2El a = fq2_mul_fq(Fq2::mul(r->x, r->y), two_inv);
  const Fq2El b = Fq2::sqr(r->y), c = Fq2::sqr(r->z);
  const Fq2El e = Fq2::mul(Fq2El{four, four}, Fq2::add(Fq2::dbl(c), c));
  const Fq2El f = Fq2::add(Fq2::dbl(e), e);
  const Fq2El g = fq2_mul_fq(Fq2::add(b, f), two_inv);
  const Fq2El h = Fq2::sub(Fq2::sqr(Fq2::add(r->y, r->z)), Fq2::add(b, c));
  const Fq2El i = Fq2::sub(e, b);
  const Fq2El j = Fq2::sqr(r->x);
  const Fq2El e2 = Fq2::sqr(e);
  r->x = Fq2::mul(a, Fq2::sub(b, f));
  r->y = Fq2::sub(Fq2::sqr(g), Fq2::add(Fq2::dbl(e2), e2));
  r->z = Fq2::mul(b, h);
  return LineCoeffs{i, Fq2::add(Fq2::dbl(j), j), Fq2::neg(h)};
}
inline B2Z_HD_NOINLINE LineCoeffs line_add(G2Homog* r, const AffinePoint<Fq2>& q) {
  const Fq2El theta = Fq2::sub(r->y, Fq2::mul(q.y, r->z));
  const Fq2El lambda = Fq2::sub(r->x, Fq2::mul(q.x, r->z));
  const Fq2El c = Fq2::sqr(theta), d = Fq2::sqr(lambda);
  const Fq2El e = Fq2::mul(lambda, d), f = Fq2::mul(r->z, c), g = Fq2::mul(r->x, d);
  const Fq2El h = Fq2::sub(Fq2::add(e, f), Fq2::dbl(g));
  r->x = Fq2::mul(lambda, h);
  r->y = Fq2::sub(Fq2::mul(theta, Fq2::sub(g, h)), Fq2::mul(e, r->y));
  r->z = Fq2::mul(r->z, e);
  const Fq2El j = Fq2::sub(Fq2::mul(theta, q.x), Fq2::mul(lambda, q.y));
  return LineCoeffs{j, Fq2::neg(theta), lambda};
}
B2Z_HD Fq12El ell(const Fq12El& f, const LineCoeffs& c, const AffinePoint<Fq>& p) {
  return fq12_mul_by_014(f, c.c0, fq2_mul_fq(c.c1, p.x), fq2_mul_fq(c.c2, p.y));
}

// ------------------------------------------------------------------ Groth16::verify_with_processed_vk, per proof
constexpr int kLines = 68;                 // 63 doubling + 5 addition steps over the bits of |x|
constexpr uint32_t kMaxInputs = 1024;

enum : uint32_t {
  PT_A_INF = 1u, PT_B_INF = 2u, PT_C_INF = 4u, PT_INPUTS_INF = 8u,
  PT_MALFORMED = 16u,                      // the single-proof verifier returns B2Z_EINVAL for this proof
};

// What the decode step hands to the Miller loop: A, B, C and the prepared inputs in affine form.
struct ProofPoints {
  AffinePoint<Fq> a, c, inputs;
  AffinePoint<Fq2> b;
  uint32_t flags;
};

// The prepared verifying key as the kernels read it (device pointers; on the host, host pointers).
struct KeyView {
  const AffinePoint<Fq>* abc;              // gamma_abc_g1, num_inputs + 1 entries
  const uint8_t* abc_inf;                  // 1 = identity
  const LineCoeffs* gamma_lines;           // kLines entries, or unused when gamma_inf
  const LineCoeffs* delta_lines;
  uint32_t num_inputs;
  uint32_t gamma_inf, delta_inf;
};

// Step 1: decode and validate A, B, C; inputs (Fr Montgomery limbs) to canonical form (>= r: malformed);
// prepared inputs = gamma_abc[0] + sum x_j gamma_abc[j + 1].
B2Z_HD void verify_decode(const uint8_t* proof, const FrEl* inputs, const KeyView& k, ProofPoints* out) {
  ProofPoints p;
  p.flags = 0;
  bool inf_a, inf_b, inf_c;
  const bool ok = g1_decompress(proof, &p.a, &inf_a) && g2_decompress(proof + 48, &p.b, &inf_b) &&
                  g1_decompress(proof + 144, &p.c, &inf_c);
  if (!ok) {
    p.flags = PT_MALFORMED;
    p.inputs = AffinePoint<Fq>{Fq::zero(), Fq::zero()};
    *out = p;
    return;
  }
  p.flags |= (inf_a ? PT_A_INF : 0u) | (inf_b ? PT_B_INF : 0u) | (inf_c ? PT_C_INF : 0u);
  G1::Xyzz acc = k.abc_inf[0] ? G1::identity() : G1::from_affine(k.abc[0]);
  uint32_t r[8];
#pragma unroll
  for (int i = 0; i < 8; i++) r[i] = FrParams::p(i);
  for (uint32_t j = 0; j < k.num_inputs; j++) {
    FrEl x = inputs[j];
    bool lt = false, decided = false;   // Montgomery limbs must be < r
#pragma unroll
    for (int i = 7; i >= 0; i--)
      if (!decided && x.l[i] != r[i]) { lt = x.l[i] < r[i]; decided = true; }
    if (!lt) {
      p.flags = PT_MALFORMED;
      *out = p;
      return;
    }
    if (k.abc_inf[j + 1]) continue;
    x = Fr::from_mont(x);
    acc = G1::add(acc, G1::mul_scalar(G1::from_affine(k.abc[j + 1]), x.l));
  }
  bool inf_p;
  p.inputs = G1::to_affine(acc, &inf_p);
  if (inf_p) p.flags |= PT_INPUTS_INF;
  *out = p;
}

// Step 2: the multi-Miller loop over (A, B), (prepared inputs, -gamma), (C, -delta); pairs with an identity point
// are skipped, as on the host.  B's lines are made on the fly, gamma's and delta's read from the key.
B2Z_HD void verify_miller(const ProofPoints& p, const KeyView& k, Fq12El* out) {
  const bool use_ab = !(p.flags & (PT_A_INF | PT_B_INF));
  const bool use_g = !(p.flags & PT_INPUTS_INF) && !k.gamma_inf;
  const bool use_d = !(p.flags & PT_C_INF) && !k.delta_inf;
  G2Homog r{p.b.x, p.b.y, Fq2::one()};
  Fq12El f = fq12_one();
  int at = 0;
  for (int i = 62; i >= 0; i--) {
    f = fq12_sqr(f);
    for (int pass = 0; pass < (((kBlsX >> i) & 1) ? 2 : 1); pass++) {
      if (use_ab) f = ell(f, pass == 0 ? line_double(&r) : line_add(&r, p.b), p.a);
      if (use_g) f = ell(f, k.gamma_lines[at], p.inputs);
      if (use_d) f = ell(f, k.delta_lines[at], p.c);
      at++;
    }
  }
  *out = fq12_conj(f);   // x < 0
}

// Step 3: final exponentiation and the comparison with alpha_g1_beta_g2; f = 0 is not valid.  Returns 1 / 0.
B2Z_HD int verify_final(const Fq12El& f, const Fq12El& alpha_beta, const FrobConsts& fc) {
  Fq12El t;
  if (!final_exponentiation(f, fc, &t)) return 0;
  return fq12_eq(t, alpha_beta) ? 1 : 0;
}

}  // namespace pairing
}  // namespace b2z
