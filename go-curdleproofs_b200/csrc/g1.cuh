// BLS12-381 G1 group law: y^2 = x^3 + 4 over Fp.
//
// Replaces gnark-crypto's G1Affine / G1Jac / g1JacExtended arithmetic that the
// reference calls at every site in SURVEY.md §8a (e.g. AddAssign
// curdleproof.go:79, ScalarMultiplication common/util.go:57, FromJacobian
// curdleproof.go:159).  Memory layouts are gnark's: G1Affine = {X, Y} (96 B,
// infinity == (0,0)), G1Jac = {X, Y, Z} (144 B, infinity == Z = 0).
//   * Jacobian coordinates carry the long doubling chains of scalar
//     multiplication (dbl 2M+5S, mixed add 8M+3S),
//   * extended Jacobian XYZZ carries MSM buckets (mixed add 8M+2S, add 12M+2S).
// Every formula handles the exceptional cases (infinity operands, P+P, P-P)
// completely: degenerate inputs do occur on this path (infinity padding in
// T'/U' curdleproof.go:156-165, all-equal MSM scalars
// samepermutationargument.go:62-67).
#pragma once
#include "fields.cuh"
#include "glv.cuh"

namespace cdl {

struct G1Affine { Fp x, y; };
struct G1Jac { Fp x, y, z; };
struct G1Xyzz { Fp x, y, zz, zzz; };

CDL_HD bool aff_is_inf(const G1Affine& p) { return FpM::is_zero(p.x) && FpM::is_zero(p.y); }
CDL_HD void aff_set_inf(G1Affine& p) { FpM::set_zero(p.x); FpM::set_zero(p.y); }
CDL_HD bool jac_is_inf(const G1Jac& p) { return FpM::is_zero(p.z); }
CDL_HD void jac_set_inf(G1Jac& p) { FpM::set_one(p.x); FpM::set_one(p.y); FpM::set_zero(p.z); }
CDL_HD bool xyzz_is_inf(const G1Xyzz& p) { return FpM::is_zero(p.zz); }
CDL_HD void xyzz_set_inf(G1Xyzz& p) {
  FpM::set_one(p.x); FpM::set_one(p.y); FpM::set_zero(p.zz); FpM::set_zero(p.zzz);
}

CDL_HD void jac_from_affine(G1Jac& r, const G1Affine& p) {
  if (aff_is_inf(p)) { jac_set_inf(r); return; }
  r.x = p.x; r.y = p.y; FpM::set_one(r.z);
}

CDL_HD void aff_neg(G1Affine& r, const G1Affine& p) { r.x = p.x; FpM::neg(r.y, p.y); }

// y^2 == x^3 + 4 (infinity (0,0) counts as on-curve, as in gnark IsOnCurve for the identity)
CDL_FN bool aff_on_curve(const G1Affine& p) {
  if (aff_is_inf(p)) return true;
  Fp l, r, b;
  FpM::sqr(l, p.y);
  FpM::sqr(r, p.x);
  FpM::mul(r, r, p.x);
  fp_set_b(b);
  FpM::add(r, r, b);
  return FpM::eq(l, r);
}

// ---------------------------------------------------------------- Jacobian
// dbl-2009-l, a = 0.  Z = 0 stays Z = 0.
CDL_FN void jac_dbl(G1Jac& r, const G1Jac& p) {
  Fp A, B, C, D, E, F, t;
  FpM::sqr(A, p.x);
  FpM::sqr(B, p.y);
  FpM::sqr(C, B);
  FpM::add(t, p.x, B);
  FpM::sqr(t, t);
  FpM::sub(t, t, A);
  FpM::sub(t, t, C);
  FpM::dbl(D, t);
  FpM::dbl(E, A);
  FpM::add(E, E, A);
  FpM::sqr(F, E);
  FpM::mul(t, p.y, p.z);  // before r.y is overwritten (r may alias p)
  FpM::dbl(r.z, t);
  FpM::dbl(t, D);
  FpM::sub(r.x, F, t);
  FpM::sub(t, D, r.x);
  FpM::mul(t, E, t);
  FpM::dbl(C, C);
  FpM::dbl(C, C);
  FpM::dbl(C, C);
  FpM::sub(r.y, t, C);
}

// r = p + q, q affine.  r may alias p.
CDL_FN void jac_add_mixed(G1Jac& r, const G1Jac& p, const G1Affine& q) {
  if (aff_is_inf(q)) { r = p; return; }
  if (jac_is_inf(p)) { r.x = q.x; r.y = q.y; FpM::set_one(r.z); return; }
  Fp z1z1, u2, s2, h, rr, hh, hhh, v, t;
  FpM::sqr(z1z1, p.z);
  FpM::mul(u2, q.x, z1z1);
  FpM::mul(s2, p.z, z1z1);
  FpM::mul(s2, s2, q.y);
  FpM::sub(h, u2, p.x);
  FpM::sub(rr, s2, p.y);
  if (FpM::is_zero(h)) {
    if (FpM::is_zero(rr)) { jac_dbl(r, p); return; }
    jac_set_inf(r);
    return;
  }
  FpM::sqr(hh, h);
  FpM::mul(hhh, hh, h);
  FpM::mul(v, p.x, hh);
  FpM::mul(r.z, p.z, h);
  FpM::sqr(t, rr);
  FpM::sub(t, t, hhh);
  FpM::sub(t, t, v);
  FpM::sub(t, t, v);       // X3
  FpM::sub(v, v, t);
  FpM::mul(v, v, rr);
  FpM::mul(hhh, hhh, p.y);
  FpM::sub(r.y, v, hhh);
  r.x = t;
}

// r = p + q, both Jacobian.  r may alias p or q.
CDL_FN void jac_add(G1Jac& r, const G1Jac& p, const G1Jac& q) {
  if (jac_is_inf(q)) { r = p; return; }
  if (jac_is_inf(p)) { r = q; return; }
  Fp z1z1, z2z2, u1, u2, s1, s2, h, rr, hh, hhh, v, t;
  FpM::sqr(z1z1, p.z);
  FpM::sqr(z2z2, q.z);
  FpM::mul(u1, p.x, z2z2);
  FpM::mul(u2, q.x, z1z1);
  FpM::mul(s1, q.z, z2z2);
  FpM::mul(s1, s1, p.y);
  FpM::mul(s2, p.z, z1z1);
  FpM::mul(s2, s2, q.y);
  FpM::sub(h, u2, u1);
  FpM::sub(rr, s2, s1);
  if (FpM::is_zero(h)) {
    if (FpM::is_zero(rr)) { jac_dbl(r, p); return; }
    jac_set_inf(r);
    return;
  }
  FpM::sqr(hh, h);
  FpM::mul(hhh, hh, h);
  FpM::mul(v, u1, hh);
  FpM::mul(t, p.z, q.z);
  FpM::mul(r.z, t, h);
  FpM::sqr(t, rr);
  FpM::sub(t, t, hhh);
  FpM::sub(t, t, v);
  FpM::sub(t, t, v);
  FpM::sub(v, v, t);
  FpM::mul(v, v, rr);
  FpM::mul(hhh, hhh, s1);
  FpM::sub(r.y, v, hhh);
  r.x = t;
}

CDL_HD void jac_neg(G1Jac& r, const G1Jac& p) { r.x = p.x; FpM::neg(r.y, p.y); r.z = p.z; }

// Jacobian -> affine with a caller-provided 1/Z (batch inversion) ...
CDL_FN void jac_to_affine_with_zinv(G1Affine& r, const G1Jac& p, const Fp& zinv) {
  if (jac_is_inf(p)) { aff_set_inf(r); return; }
  Fp zi2, zi3;
  FpM::sqr(zi2, zinv);
  FpM::mul(zi3, zi2, zinv);
  FpM::mul(r.x, p.x, zi2);
  FpM::mul(r.y, p.y, zi3);
}
// ... or with its own field inversion.
CDL_FN void jac_to_affine(G1Affine& r, const G1Jac& p) {
  Fp zi;
  fp_inv(zi, p.z);
  jac_to_affine_with_zinv(r, p, zi);
}

// p == q as group elements (cross-multiplied, no inversion)
CDL_FN bool jac_eq(const G1Jac& p, const G1Jac& q) {
  bool pi = jac_is_inf(p), qi = jac_is_inf(q);
  if (pi || qi) return pi && qi;
  Fp z1z1, z2z2, a, b;
  FpM::sqr(z1z1, p.z);
  FpM::sqr(z2z2, q.z);
  FpM::mul(a, p.x, z2z2);
  FpM::mul(b, q.x, z1z1);
  if (!FpM::eq(a, b)) return false;
  FpM::mul(z1z1, z1z1, p.z);
  FpM::mul(z2z2, z2z2, q.z);
  FpM::mul(a, p.y, z2z2);
  FpM::mul(b, q.y, z1z1);
  return FpM::eq(a, b);
}

// ---------------------------------------------------------------- XYZZ
// mdbl-2008-s-1: r = 2q, q affine (not infinity)
CDL_FN void xyzz_dbl_affine(G1Xyzz& r, const G1Affine& q) {
  Fp u, s, m, t;
  FpM::dbl(u, q.y);
  FpM::sqr(r.zz, u);            // V
  FpM::mul(r.zzz, u, r.zz);     // W
  FpM::mul(s, q.x, r.zz);
  FpM::sqr(m, q.x);
  FpM::dbl(t, m);
  FpM::add(m, m, t);            // 3 X^2
  FpM::sqr(r.x, m);
  FpM::sub(r.x, r.x, s);
  FpM::sub(r.x, r.x, s);
  FpM::sub(s, s, r.x);
  FpM::mul(s, s, m);
  FpM::mul(t, r.zzz, q.y);
  FpM::sub(r.y, s, t);
}

// dbl-2008-s-1: r = 2p.  r may alias p.
CDL_FN void xyzz_dbl(G1Xyzz& r, const G1Xyzz& p) {
  if (xyzz_is_inf(p)) { r = p; return; }
  Fp u, v, w, s, m, t;
  FpM::dbl(u, p.y);
  FpM::sqr(v, u);
  FpM::mul(w, u, v);
  FpM::mul(s, p.x, v);
  FpM::sqr(m, p.x);
  FpM::dbl(t, m);
  FpM::add(m, m, t);
  FpM::mul(t, w, p.y);          // W*Y1 before r.y changes
  FpM::mul(r.zz, v, p.zz);
  FpM::mul(r.zzz, w, p.zzz);
  FpM::sqr(u, m);
  FpM::sub(u, u, s);
  FpM::sub(u, u, s);            // X3
  FpM::sub(s, s, u);
  FpM::mul(s, s, m);
  FpM::sub(r.y, s, t);
  r.x = u;
}

// madd-2008-s: r = p + q, q affine.  r may alias p.
CDL_FN void xyzz_add_mixed(G1Xyzz& r, const G1Xyzz& p, const G1Affine& q) {
  if (aff_is_inf(q)) { r = p; return; }
  if (xyzz_is_inf(p)) { r.x = q.x; r.y = q.y; FpM::set_one(r.zz); FpM::set_one(r.zzz); return; }
  Fp u2, s2, pp, ppp, qq, t;
  FpM::mul(u2, q.x, p.zz);
  FpM::mul(s2, q.y, p.zzz);
  FpM::sub(u2, u2, p.x);        // P
  FpM::sub(s2, s2, p.y);        // R
  if (FpM::is_zero(u2)) {
    if (FpM::is_zero(s2)) { xyzz_dbl_affine(r, q); return; }
    xyzz_set_inf(r);
    return;
  }
  FpM::sqr(pp, u2);
  FpM::mul(ppp, pp, u2);
  FpM::mul(qq, p.x, pp);
  FpM::mul(r.zz, p.zz, pp);
  FpM::mul(r.zzz, p.zzz, ppp);
  FpM::sqr(t, s2);
  FpM::sub(t, t, ppp);
  FpM::sub(t, t, qq);
  FpM::sub(t, t, qq);           // X3
  FpM::sub(qq, qq, t);
  FpM::mul(qq, qq, s2);
  FpM::mul(ppp, ppp, p.y);
  FpM::sub(r.y, qq, ppp);
  r.x = t;
}

// add-2008-s: r = p + q.  r may alias p or q.
CDL_FN void xyzz_add(G1Xyzz& r, const G1Xyzz& p, const G1Xyzz& q) {
  if (xyzz_is_inf(q)) { r = p; return; }
  if (xyzz_is_inf(p)) { r = q; return; }
  Fp u1, u2, s1, s2, pp, ppp, qq, t;
  FpM::mul(u1, p.x, q.zz);
  FpM::mul(u2, q.x, p.zz);
  FpM::mul(s1, p.y, q.zzz);
  FpM::mul(s2, q.y, p.zzz);
  FpM::sub(u2, u2, u1);         // P
  FpM::sub(s2, s2, s1);         // R
  if (FpM::is_zero(u2)) {
    if (FpM::is_zero(s2)) { xyzz_dbl(r, p); return; }
    xyzz_set_inf(r);
    return;
  }
  FpM::sqr(pp, u2);
  FpM::mul(ppp, pp, u2);
  FpM::mul(qq, u1, pp);
  FpM::mul(t, p.zz, q.zz);
  FpM::mul(r.zz, t, pp);
  FpM::mul(t, p.zzz, q.zzz);
  FpM::mul(r.zzz, t, ppp);
  FpM::sqr(t, s2);
  FpM::sub(t, t, ppp);
  FpM::sub(t, t, qq);
  FpM::sub(t, t, qq);
  FpM::sub(qq, qq, t);
  FpM::mul(qq, qq, s2);
  FpM::mul(ppp, ppp, s1);
  FpM::sub(r.y, qq, ppp);
  r.x = t;
}

// XYZZ -> Jacobian without inversion: (X, Y, ZZ, ZZZ) ~ (X*ZZZ^2*ZZ^2..)...
// Use Z = ZZZ/ZZ-free form: (X*ZZ, Y*ZZZ, ZZ) is Jacobian with Z' = ZZ:
//   X'/Z'^2 = X*ZZ/ZZ^2 = X/ZZ,  Y'/Z'^3 = Y*ZZZ/ZZ^3 = Y/ZZZ (since ZZ^3 = ZZZ^2).
CDL_HD void xyzz_to_jac(G1Jac& r, const G1Xyzz& p) {
  if (xyzz_is_inf(p)) { jac_set_inf(r); return; }
  FpM::mul(r.x, p.x, p.zz);
  FpM::mul(r.y, p.y, p.zzz);
  r.z = p.zz;
}

CDL_HD void xyzz_from_affine(G1Xyzz& r, const G1Affine& q) {
  if (aff_is_inf(q)) { xyzz_set_inf(r); return; }
  r.x = q.x; r.y = q.y; FpM::set_one(r.zz); FpM::set_one(r.zzz);
}

CDL_HD void xyzz_neg(G1Xyzz& r, const G1Xyzz& p) { r = p; FpM::neg(r.y, p.y); }

// ---------------------------------------------------------------- scalar mul
// Signed fixed-window recoding of a canonical 256-bit scalar (k < 2^255):
// k = sum d_i 16^i, d_i in [-8, 8], 64 digits.  Uniform schedule: every lane of
// a warp performs the same doublings/additions regardless of its scalar.
CDL_HD void recode_w4(int8_t* digits, const uint32_t* k) {
  uint32_t carry = 0;
  for (int i = 0; i < 64; i++) {
    uint32_t d = ((k[i >> 3] >> ((i & 7) * 4)) & 15u) + carry;
    carry = d > 8u;
    digits[i] = (int8_t)((int)d - (int)(carry << 4));
  }
}

// r = k * p, k canonical (non-Montgomery) little-endian words, k < 2^255.  Plain signed-window form without
// the GLV split: the CPU tier (tests/hostcheck) uses it as the independent cross-check of jac_scalar_mul_glv.
CDL_FN void jac_scalar_mul(G1Jac& r, const G1Affine& p, const uint32_t* k) {
  if (aff_is_inf(p)) { jac_set_inf(r); return; }
  G1Jac tab[8];  // tab[i] = (i+1) p
  jac_from_affine(tab[0], p);
  jac_dbl(tab[1], tab[0]);
#pragma unroll 1
  for (int i = 2; i < 8; i++) jac_add_mixed(tab[i], tab[i - 1], p);
  int8_t dg[64];
  recode_w4(dg, k);
  jac_set_inf(r);
#pragma unroll 1
  for (int i = 63; i >= 0; i--) {
    if (i != 63) {
#pragma unroll 1
      for (int j = 0; j < 4; j++) jac_dbl(r, r);
    }
    int d = dg[i];
    if (d != 0) {
      int a = d < 0 ? -d : d;
      G1Jac t = tab[a - 1];
      if (d < 0) FpM::neg(t.y, t.y);
      jac_add(r, r, t);
    }
  }
}


// General-case mixed addition that also returns H = U2 - X1 (Z3 = Z1 * H): the ratio
// between consecutive Z coordinates of a table built by repeated addition.  No exceptional
// cases: callers only add P to i*P (1 < i < 8) for P of prime order.
CDL_FN void jac_add_mixed_h(G1Jac& r, const G1Jac& p, const G1Affine& q, Fp& h) {
  Fp z1z1, u2, s2, rr, hh, hhh, v, t;
  FpM::sqr(z1z1, p.z);
  FpM::mul(u2, q.x, z1z1);
  FpM::mul(s2, p.z, z1z1);
  FpM::mul(s2, s2, q.y);
  FpM::sub(h, u2, p.x);
  FpM::sub(rr, s2, p.y);
  FpM::sqr(hh, h);
  FpM::mul(hhh, hh, h);
  FpM::mul(v, p.x, hh);
  FpM::mul(r.z, p.z, h);
  FpM::sqr(t, rr);
  FpM::sub(t, t, hhh);
  FpM::sub(t, t, v);
  FpM::sub(t, t, v);
  FpM::sub(v, v, t);
  FpM::mul(v, v, rr);
  FpM::mul(hhh, hhh, p.y);
  FpM::sub(r.y, v, hhh);
  r.x = t;
}

// r = k * p via GLV: k = s0*(s1*|k1| + k2*lambda), phi(p) = (beta*x, y) = lambda*p.
// 32 signed 4-bit windows, 4 doublings + up to 2 additions per window.  Same uniform
// schedule for every lane.  k canonical little-endian words, k < r; p of prime order.
//
// The window table {1..8}P is brought to a COMMON Z without an inversion: built by repeated
// addition its Z coordinates satisfy Z_{i+1} = Z_i * H_i, so entry i times (Z_8 / Z_i)^2,
// (Z_8 / Z_i)^3 is the affine form of i*P on the isomorphic curve y^2 = x^3 + 4*Z_8^6.  The
// doubling and mixed-addition formulas do not involve the curve constant, so the whole
// multiplication runs on that curve with MIXED additions (11 instead of 16 products each,
// and phi is still (beta*x, y) there); the result maps back by Z <- Z * Z_8.
CDL_FN void jac_scalar_mul_glv(G1Jac& r, const G1Affine& p, const uint32_t* k) {
  if (aff_is_inf(p)) { jac_set_inf(r); return; }
  Glv g;
  glv_decompose(g, k);
  G1Affine tab[8];  // tab[i] = (i+1) p on the isomorphic curve
  Fp zc;            // common Z = Z of 8p
  {
    G1Jac acc, first;
    Fp h[8];        // h[i] = Z_{i+1} / Z_i for the additions producing entries 2..7 (0-based)
    jac_from_affine(first, p);
    jac_dbl(acc, first);
    tab[1].x = acc.x; tab[1].y = acc.y;
    Fp z2 = acc.z;
#pragma unroll 1
    for (int i = 2; i < 8; i++) {
      jac_add_mixed_h(acc, acc, p, h[i]);
      tab[i].x = acc.x; tab[i].y = acc.y;
    }
    zc = acc.z;
    // s = Z_8 / Z_{i+1}: running product of the later ratios
    Fp sfac;
    FpM::set_one(sfac);
#pragma unroll 1
    for (int i = 6; i >= 0; i--) {
      if (i >= 1) FpM::mul(sfac, sfac, h[i + 1]);  // entries 2..7 (index 1..6): s_i = prod_{j>i} h_j
      else FpM::mul(sfac, sfac, z2);                // entry 1: Z_1 = 1, s = Z_8 = Z_2 * prod h
      Fp s2, s3;
      FpM::sqr(s2, sfac);
      FpM::mul(s3, s2, sfac);
      if (i >= 1) {
        FpM::mul(tab[i].x, tab[i].x, s2);
        FpM::mul(tab[i].y, tab[i].y, s3);
      } else {
        FpM::mul(tab[0].x, p.x, s2);
        FpM::mul(tab[0].y, p.y, s3);
      }
    }
  }
  int8_t dg[2][32];
  recode_w4_128(dg[0], g.k1);
  recode_w4_128(dg[1], g.k2);
  Fp beta;
  fp_set_beta(beta);
  jac_set_inf(r);
#pragma unroll 1
  for (int i = 31; i >= 0; i--) {
    if (i != 31) {
#pragma unroll 1
      for (int j = 0; j < 4; j++) jac_dbl(r, r);
    }
#pragma unroll 1
    for (int h = 0; h < 2; h++) {
      int d = dg[h][i];
      if (d != 0) {
        int a = d < 0 ? -d : d;
        G1Affine t = tab[a - 1];
        if (h == 1) FpM::mul(t.x, t.x, beta);
        bool neg = (d < 0) != (h == 0 ? g.neg1 : g.neg2);
        if (neg) FpM::neg(t.y, t.y);
        jac_add_mixed(r, r, t);
      }
    }
  }
  FpM::mul(r.z, r.z, zc);  // back from the isomorphic curve (infinity stays Z = 0)
}

CDL_FN void jac_dbl_n(G1Jac& r, int n) {
#pragma unroll 1
  for (int i = 0; i < n; i++) jac_dbl(r, r);
}

// Subgroup membership by the endomorphism: P is in G1 iff P + [z^2] phi(P) = 0, i.e. [z^2] phi(P) = -P
// (z^2 * lambda + 1 = r).  This is gnark-crypto's own G1 IsInSubGroup test (126 doublings + 10 additions
// instead of a 255-bit multiplication by r).  z^2 phi(P) is computed as |z| (|z| phi(P)).  |z| =
// 0xd201000000010000 has bits 63, 62, 60, 57, 48 and 16 set: from the top bit, the doubling runs 1, 2, 3, 9, 32
// each end in an addition of the base, then 16 doublings follow.  The first base, phi(P) = (beta x, y), is
// affine, so its additions are mixed; the second, |z| phi(P), stays Jacobian (normalising it would cost an
// inversion).  Every addition keeps the complete exceptional-case handling: P need not have prime order here.
CDL_FN bool g1_in_subgroup_endo(const G1Affine& p) {
  if (aff_is_inf(p)) return true;
  constexpr uint32_t kRuns = 1u | 2u << 6 | 3u << 12 | 9u << 18 | 32u << 24;  // 6 bits per run
  G1Affine q;
  Fp beta;
  fp_set_beta(beta);
  FpM::mul(q.x, p.x, beta);
  q.y = p.y;
  G1Jac t, u;
  jac_from_affine(t, q);
#pragma unroll 1
  for (int s = 0; s < 30; s += 6) {
    jac_dbl_n(t, (kRuns >> s) & 63u);
    jac_add_mixed(t, t, q);
  }
  jac_dbl_n(t, 16);
  u = t;
#pragma unroll 1
  for (int s = 0; s < 30; s += 6) {
    jac_dbl_n(t, (kRuns >> s) & 63u);
    jac_add(t, t, u);
  }
  jac_dbl_n(t, 16);
  // t == -P without normalising t: X = x Z^2 and Y = -y Z^3.  t = infinity is never -P (P is finite).
  if (jac_is_inf(t)) return false;
  Fp zz, w;
  FpM::sqr(zz, t.z);
  FpM::mul(w, p.x, zz);
  if (!FpM::eq(w, t.x)) return false;
  FpM::mul(zz, zz, t.z);
  FpM::mul(w, p.y, zz);
  FpM::add(w, w, t.y);
  return FpM::is_zero(w);
}

}  // namespace cdl
