// BN254 G1 (over Fq) and G2 (over Fq2 = Fq[u]/(u^2+1)) group arithmetic, templated over the coordinate field.
//
// Replaces (upstream, not vendored: yarn.lock:408-416, 1132-1135) ffjavascript src/f2field.js + src/ec.js and
// wasmcurves build_curve_jacobian_a0.js (g1m_* / g2m_* add, double, affine conversion).  The WASM code works in
// Jacobian coordinates; here bucket accumulators are extended-Jacobian "XYZZ" (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2)
// because the mixed addition is 8M+2S and needs no inversion.  Group elements are exact, so the affine result
// of any sum is bit-identical to the reference's whatever coordinate system produced it.
//
// Affine buffers follow the zkey convention (SURVEY.md 8b): Montgomery coordinates, (0,0) = point at infinity.
#pragma once
#include "fp.cuh"

namespace nzcp {

// ------------------------------------------------------------------------------------------------ Fq2
struct Fq2 {
  Fq c0, c1;
  HD static Fq2 zero() { return Fq2{Fq::zero(), Fq::zero()}; }
  HD static Fq2 one() { return Fq2{Fq::one(), Fq::zero()}; }
  HD bool is_zero() const { return c0.is_zero() && c1.is_zero(); }
  HD bool operator==(const Fq2& b) const { return c0 == b.c0 && c1 == b.c1; }
  HD bool operator!=(const Fq2& b) const { return !(*this == b); }
};

// uniform free-function interface over Fq and Fq2
HD Fq f_add(const Fq& a, const Fq& b) { return fp_add(a, b); }
HD Fq f_sub(const Fq& a, const Fq& b) { return fp_sub(a, b); }
HD Fq f_mul(const Fq& a, const Fq& b) { return fp_mul(a, b); }
HD Fq f_sqr(const Fq& a) { return fp_sqr(a); }
HD Fq f_neg(const Fq& a) { return fp_neg(a); }
HD Fq f_dbl(const Fq& a) { return fp_add(a, a); }
HDN inline Fq f_inv(const Fq& a) { return fp_inv(a); }
HD Fq f_from_mont(const Fq& a) { return fp_from_mont(a); }

HD Fq2 f_add(const Fq2& a, const Fq2& b) { return Fq2{fp_add(a.c0, b.c0), fp_add(a.c1, b.c1)}; }
HD Fq2 f_sub(const Fq2& a, const Fq2& b) { return Fq2{fp_sub(a.c0, b.c0), fp_sub(a.c1, b.c1)}; }
HD Fq2 f_neg(const Fq2& a) { return Fq2{fp_neg(a.c0), fp_neg(a.c1)}; }
HD Fq2 f_dbl(const Fq2& a) { return Fq2{fp_add(a.c0, a.c0), fp_add(a.c1, a.c1)}; }
// On the device an Fq2 product / square is a real function call: a G2 mixed addition is 28 Fq products, and inlining
// all of them (~6 000 SASS instructions) made the G2 bucket-accumulate kernel stall on instruction fetch (ncu:
// stalled_no_instruction ~3 per issue).  Two shared bodies (3 and 2 Fq products) stay resident in the i-cache; calling
// at Fq2 granularity moves 48 registers per 3 products instead of 24 per product.
HD Fq2 f2_mul_inline(const Fq2& a, const Fq2& b) {  // Karatsuba, 3 Fq mul; u^2 = -1
  Fq t0 = fp_mul(a.c0, b.c0);
  Fq t1 = fp_mul(a.c1, b.c1);
  Fq t2 = fp_mul(fp_add(a.c0, a.c1), fp_add(b.c0, b.c1));
  return Fq2{fp_sub(t0, t1), fp_sub(fp_sub(t2, t0), t1)};
}
HD Fq2 f2_sqr_inline(const Fq2& a) {  // (c0+c1)(c0-c1) + 2 c0 c1 u : 2 Fq mul
  Fq t0 = fp_mul(fp_add(a.c0, a.c1), fp_sub(a.c0, a.c1));
  Fq t1 = fp_mul(a.c0, a.c1);
  return Fq2{t0, fp_add(t1, t1)};
}
#if !defined(NZCP_FQ2_NO_LAZY) && !defined(NZCP_FQ2_LAZY)
#define NZCP_FQ2_LAZY 1   // default on: bit-exact (full GPU suite), G2 kernels 4-15 % faster
#endif
#if defined(__CUDA_ARCH__) && defined(NZCP_FQ2_LAZY)
// Lazy reduction: the three Karatsuba products stay 512-bit integers and only the two results are Montgomery-reduced:
// 3 wide products + 2 reductions = 320 32x32 products instead of 3 x 128 = 384.
//   c1 = REDC((a0+a1)(b0+b1) - a0 b0 - a1 b1)          (>= 0, < 2 p^2)
//   c0 = REDC(a0 b0 - a1 b1 + p^2)                      (> 0,  < 2 p^2)
__device__ __forceinline__ Fq2 f2_mul_lazy(const Fq2& a, const Fq2& b) {
  const uint32_t P2[16] = {0x275d69b1u, 0x3b5458a2u, 0x09eac101u, 0xa602072du, 0x6d96cadcu, 0x4a50189cu, 0x7a1242c8u, 0x04689e95u,
                           0x34c6b38du, 0x26edfa5cu, 0x16375606u, 0xb00b8551u, 0x0348d21cu, 0x599a6f7cu, 0x763cbf9cu, 0x0925c4b8u};
  uint32_t T0[16], T1[16], T2[16], sa[8], sb[8];
  fp_mul_wide(T0, a.c0.v, b.c0.v);
  fp_mul_wide(T1, a.c1.v, b.c1.v);
  fp_add8c(sa, a.c0.v, a.c1.v, 0u);   // < 2^255: no reduction needed before the product
  fp_add8c(sb, b.c0.v, b.c1.v, 0u);
  fp_mul_wide(T2, sa, sb);
  fp_sub16(T2, T2, T0);
  fp_sub16(T2, T2, T1);
  fp_add16(T0, T0, P2);
  fp_sub16(T0, T0, T1);
  Fq2 r;
  fp_redc_wide<FqParams>(r.c0.v, T0);
  fp_redc_wide<FqParams>(r.c1.v, T2);
  return r;
}
#endif
#if defined(__CUDA_ARCH__) && !defined(NZCP_FQ2_INLINE)
#if defined(NZCP_FQ2_LAZY)
__device__ __noinline__ Fq2 f2_mul_call(Fq2 a, Fq2 b) { return f2_mul_lazy(a, b); }
#else
__device__ __noinline__ Fq2 f2_mul_call(Fq2 a, Fq2 b) { return f2_mul_inline(a, b); }
#endif
__device__ __noinline__ Fq2 f2_sqr_call(Fq2 a) { return f2_sqr_inline(a); }
HD Fq2 f_mul(const Fq2& a, const Fq2& b) { return f2_mul_call(a, b); }
HD Fq2 f_sqr(const Fq2& a) { return f2_sqr_call(a); }
#else
HD Fq2 f_mul(const Fq2& a, const Fq2& b) { return f2_mul_inline(a, b); }
HD Fq2 f_sqr(const Fq2& a) { return f2_sqr_inline(a); }
#endif
HDN inline Fq2 f_inv(const Fq2& a) {
  Fq d = fp_inv(fp_add(fp_sqr(a.c0), fp_sqr(a.c1)));
  return Fq2{fp_mul(a.c0, d), fp_neg(fp_mul(a.c1, d))};
}
HD Fq2 f_from_mont(const Fq2& a) { return Fq2{fp_from_mont(a.c0), fp_from_mont(a.c1)}; }
// Inversion by division steps (fp.cuh fp_inv_fast): constant time, ~50 products' worth of issue slots.  0 -> 0.
HDN inline Fq f_inv_fast(const Fq& a) { return fp_inv_fast(a); }
HDN inline Fq2 f_inv_fast(const Fq2& a) {
  Fq d = fp_inv_fast(fp_add(fp_sqr(a.c0), fp_sqr(a.c1)));
  return Fq2{fp_mul(a.c0, d), fp_neg(fp_mul(a.c1, d))};
}

// a*b - c*d.  Every group-law formula ends its y coordinate with this shape (Y3 = R (Q - X3) - Y1 PPP); on the device
// the Fq version keeps both products as 512-bit integers and reduces once: 2 wide products + 1 reduction = 192 32x32
// products instead of 256.
HD Fq f_mulsub(const Fq& a, const Fq& b, const Fq& c, const Fq& d) {
#if defined(__CUDA_ARCH__) && !defined(NZCP_NO_MULSUB_LAZY)
  const uint32_t P2[16] = {0x275d69b1u, 0x3b5458a2u, 0x09eac101u, 0xa602072du, 0x6d96cadcu, 0x4a50189cu, 0x7a1242c8u, 0x04689e95u,
                           0x34c6b38du, 0x26edfa5cu, 0x16375606u, 0xb00b8551u, 0x0348d21cu, 0x599a6f7cu, 0x763cbf9cu, 0x0925c4b8u};
  uint32_t Ta[16], Tb[16];
  fp_mul_wide(Ta, a.v, b.v);
  fp_mul_wide(Tb, c.v, d.v);
  fp_add16(Ta, Ta, P2);     // + p^2 keeps the difference positive; a b - c d + p^2 < 2 p^2 < p * 2^256
  fp_sub16(Ta, Ta, Tb);
  Fq r;
  fp_redc_wide<FqParams>(r.v, Ta);
  return r;
#else
  return fp_sub(fp_mul(a, b), fp_mul(c, d));
#endif
}
HD Fq2 f_mulsub(const Fq2& a, const Fq2& b, const Fq2& c, const Fq2& d) { return f_sub(f_mul(a, b), f_mul(c, d)); }

// ------------------------------------------------------------------------------------------------ points
template <class F>
struct Affine {
  F x, y;
  HD bool is_inf() const { return x.is_zero() && y.is_zero(); }
  HD static Affine inf() { return Affine{F::zero(), F::zero()}; }
};

template <class F>
struct XYZZ {
  F x, y, zz, zzz;
  HD bool is_inf() const { return zz.is_zero(); }
  HD static XYZZ inf() { return XYZZ{F::zero(), F::zero(), F::zero(), F::zero()}; }
  HD static XYZZ from_affine(const Affine<F>& p) {
    if (p.is_inf()) return inf();
    return XYZZ{p.x, p.y, F::one(), F::one()};
  }
};

template <class F>
HD XYZZ<F> xyzz_neg(const XYZZ<F>& p) {
  return XYZZ<F>{p.x, f_neg(p.y), p.zz, p.zzz};
}

// dbl-2008-s-1 (a = 0)
template <class F>
HD XYZZ<F> xyzz_dbl(const XYZZ<F>& p) {
  if (p.is_inf()) return p;
  F u = f_dbl(p.y);
  F v = f_sqr(u);
  F w = f_mul(u, v);
  F s = f_mul(p.x, v);
  F xx = f_sqr(p.x);
  F m = f_add(f_dbl(xx), xx);
  XYZZ<F> r;
  r.x = f_sub(f_sqr(m), f_dbl(s));
  r.y = f_mulsub(m, f_sub(s, r.x), w, p.y);
  r.zz = f_mul(v, p.zz);
  r.zzz = f_mul(w, p.zzz);
  return r;
}

// Doubling of an affine point (mdbl-2008-s-1); y != 0 on these curves (no 2-torsion).
template <class F>
HD XYZZ<F> xyzz_dbl_affine(const Affine<F>& p) {
  F u = f_dbl(p.y);
  F v = f_sqr(u);
  F w = f_mul(u, v);
  F s = f_mul(p.x, v);
  F xx = f_sqr(p.x);
  F m = f_add(f_dbl(xx), xx);
  XYZZ<F> r;
  r.x = f_sub(f_sqr(m), f_dbl(s));
  r.y = f_mulsub(m, f_sub(s, r.x), w, p.y);
  r.zz = v;
  r.zzz = w;
  return r;
}

// acc += (q.x, neg ? -q.y : q.y)   madd-2008-s, 8M + 2S; q must not be infinity.
template <class F>
HD void xyzz_madd(XYZZ<F>& acc, const Affine<F>& q, bool neg) {
  F qy = neg ? f_neg(q.y) : q.y;
  if (acc.is_inf()) {
    acc.x = q.x;
    acc.y = qy;
    acc.zz = F::one();
    acc.zzz = F::one();
    return;
  }
  F u2 = f_mul(q.x, acc.zz);
  F s2 = f_mul(qy, acc.zzz);
  F p = f_sub(u2, acc.x);
  F r = f_sub(s2, acc.y);
  if (p.is_zero()) {
    if (r.is_zero()) {
      acc = xyzz_dbl_affine(Affine<F>{q.x, qy});
    } else {
      acc = XYZZ<F>::inf();
    }
    return;
  }
  F pp = f_sqr(p);
  F ppp = f_mul(p, pp);
  F qq = f_mul(acc.x, pp);
  F x3 = f_sub(f_sub(f_sqr(r), ppp), f_dbl(qq));
  acc.y = f_mulsub(r, f_sub(qq, x3), acc.y, ppp);
  acc.x = x3;
  acc.zz = f_mul(acc.zz, pp);
  acc.zzz = f_mul(acc.zzz, ppp);
}

// acc += b   add-2008-s, 12M + 2S
template <class F>
HD void xyzz_add(XYZZ<F>& acc, const XYZZ<F>& b) {
  if (b.is_inf()) return;
  if (acc.is_inf()) {
    acc = b;
    return;
  }
  F u1 = f_mul(acc.x, b.zz);
  F u2 = f_mul(b.x, acc.zz);
  F s1 = f_mul(acc.y, b.zzz);
  F s2 = f_mul(b.y, acc.zzz);
  F p = f_sub(u2, u1);
  F r = f_sub(s2, s1);
  if (p.is_zero()) {
    if (r.is_zero()) {
      acc = xyzz_dbl(acc);
    } else {
      acc = XYZZ<F>::inf();
    }
    return;
  }
  F pp = f_sqr(p);
  F ppp = f_mul(p, pp);
  F qq = f_mul(u1, pp);
  F x3 = f_sub(f_sub(f_sqr(r), ppp), f_dbl(qq));
  acc.y = f_mulsub(r, f_sub(qq, x3), s1, ppp);
  acc.x = x3;
  acc.zz = f_mul(f_mul(acc.zz, b.zz), pp);
  acc.zzz = f_mul(f_mul(acc.zzz, b.zzz), ppp);
}

// k * p, k = plain 256-bit little-endian scalar (8 limbs); left-to-right with a 4-bit window (table of 1..15 times p).
template <class F>
HDN inline XYZZ<F> xyzz_mul(const XYZZ<F>& p, const uint32_t* k) {
  XYZZ<F> tab[16];
  tab[0] = XYZZ<F>::inf();
  tab[1] = p;
  for (int i = 2; i < 16; i++) {
    tab[i] = tab[i - 1];
    xyzz_add(tab[i], p);
  }
  XYZZ<F> r = XYZZ<F>::inf();
  for (int i = 63; i >= 0; i--) {
    if (!r.is_inf())
      for (int d = 0; d < 4; d++) r = xyzz_dbl(r);
    uint32_t nib = (k[i >> 3] >> ((i & 7) * 4)) & 15;
    if (nib) xyzz_add(r, tab[nib]);
  }
  return r;
}

// Bits pos .. pos+4 of a 256-bit little-endian scalar; bits below 0 read as 0.
HD uint32_t scalar_bits5(const uint32_t* v, int pos) {
  if (pos < 0) return (v[0] << 1) & 31u;
  const int l = pos >> 5;
  uint64_t w = v[l];
  if (l < 7) w |= (uint64_t)v[l + 1] << 32;
  return (uint32_t)(w >> (pos & 31)) & 31u;
}

// acc += k * P for an affine P and a plain scalar k < r.  k > (r-1)/2 is folded to (r - k) * (-P), so the -1 / small
// negative coefficients circom emits cost one addition.  The rest is a signed 4-bit fixed window (radix-16 Booth digits
// d_i = b(4i-1) + b(4i) + 2 b(4i+1) + 4 b(4i+2) - 8 b(4i+3), in [-8, 8]) over a table of 1..8 * P: 4 doublings and at most
// one addition per digit.  The digits of every lane of a warp fall at the same positions, so the additions do not
// diverge the way a per-bit double-and-add does (one lane or another has a set bit at almost every position).
template <class F>
HD void scalar_mul_accumulate(XYZZ<F>& acc, const Affine<F>& P, Fr k) {
  if (P.is_inf() || k.is_zero()) return;
  bool neg = false;
  {
    Fr nk = fp_sub(Fr::zero(), k);       // r - k (plain integers: canonical subtraction mod r)
    bool gt = false;
#pragma unroll
    for (int i = 7; i >= 0; i--) {
      if (k.v[i] != nk.v[i]) { gt = k.v[i] > nk.v[i]; break; }
    }
    if (gt) { k = nk; neg = true; }
  }
  int top = 255;
  while (top > 0 && !((k.v[top >> 5] >> (top & 31)) & 1)) top--;
  if (top == 0) {                        // k == 1
    xyzz_madd(acc, P, neg);
    return;
  }
  XYZZ<F> tab[8];                        // tab[j] = (j + 1) * P
  tab[0] = XYZZ<F>::from_affine(P);
  tab[1] = xyzz_dbl_affine(P);
  for (int j = 2; j < 8; j++) {
    tab[j] = tab[j - 1];
    xyzz_madd(tab[j], P, false);
  }
  XYZZ<F> r = XYZZ<F>::inf();
  for (int i = (top + 1) >> 2; i >= 0; i--) {   // k < r/2 < 2^253: no digit above bit 252 + 1
    for (int d = 0; d < 4; d++) r = xyzz_dbl(r);
    const uint32_t w = scalar_bits5(k.v, 4 * i - 1);
    const int d = (int)((w + 1) >> 1) - (int)((w >> 4) << 4);
    if (d) {
      XYZZ<F> t = tab[(d < 0 ? -d : d) - 1];
      if (d < 0) t = xyzz_neg(t);
      xyzz_add(r, t);
    }
  }
  if (neg) r = xyzz_neg(r);
  xyzz_add(acc, r);
}

// Curve membership of an affine point in Montgomery form: canonical coordinates and y^2 = x^3 + b, or the (0,0) marker.
template <class F> struct CoordCanon;
template <> struct CoordCanon<Fq> {
  HD static bool ok(const Fq& a) { return !fp_geq_mod<FqParams>(a.v); }
};
template <> struct CoordCanon<Fq2> {
  HD static bool ok(const Fq2& a) { return !fp_geq_mod<FqParams>(a.c0.v) && !fp_geq_mod<FqParams>(a.c1.v); }
};

template <class F>
HD bool point_ok(const Affine<F>& p, const F& b, bool* inf) {
  *inf = p.is_inf();
  if (*inf) return true;
  if (!CoordCanon<F>::ok(p.x) || !CoordCanon<F>::ok(p.y)) return false;
  const F lhs = f_sqr(p.y);
  const F rhs = f_add(f_mul(f_sqr(p.x), p.x), b);
  return lhs == rhs;
}

template <class F>
HD F curve_b(const Affine<F>& gen) {   // b = y^2 - x^3 of the generator (Montgomery form)
  return f_sub(f_sqr(gen.y), f_mul(f_sqr(gen.x), gen.x));
}

// Montgomery-form affine; infinity -> (0,0).
template <class F>
HDN inline Affine<F> xyzz_to_affine(const XYZZ<F>& p) {
  if (p.is_inf()) return Affine<F>::inf();
  F iz3 = f_inv(p.zzz);               // 1/Z^3
  F iz2 = f_sqr(f_mul(iz3, p.zz));    // (Z^2/Z^3)^2 = 1/Z^2
  return Affine<F>{f_mul(p.x, iz2), f_mul(p.y, iz3)};
}

// Montgomery-form affine through the division-step inversion (fp_inv_fast): the per-point conversion of the kernels that
// write one affine point per thread.
template <class F>
HD Affine<F> to_affine_fast(const XYZZ<F>& p) {
  if (p.is_inf()) return Affine<F>::inf();
  const F iz3 = f_inv_fast(p.zzz);
  const F iz2 = f_sqr(f_mul(iz3, p.zz));
  return Affine<F>{f_mul(p.x, iz2), f_mul(p.y, iz3)};
}

typedef Affine<Fq> G1Affine;
typedef Affine<Fq2> G2Affine;
typedef XYZZ<Fq> G1XYZZ;
typedef XYZZ<Fq2> G2XYZZ;

}  // namespace nzcp
