// BN254 G1 (y^2 = x^3 + 3 over Fq) group law for the MSM kernels.
//
// Replaces py_ecc.bn128 `add` / `double` (one Fq inversion per operation; SURVEY App. A) as used by
// curve.py:38-111 `ec_lincomb`.  Accumulators use extended Jacobian "XYZZ" coordinates
// (x = X/ZZ, y = Y/ZZZ, ZZ^3 = ZZZ^2; identity <=> ZZ == 0) so an affine point is added with
// 8 mul + 2 sqr and no inversion; a single inversion happens in g1_to_affine at the very end.
// Formulas: the standard madd-2008-s / add-2008-s / dbl-2008-s-1 sets for short Weierstrass curves
// with a = 0.  Their Y3 = A B - C D is computed as (A B + C (p - D)) R^-1 with one Montgomery
// reduction for both products (fp_mul_sum2), and squarings use fp_sqr, so an affine addition costs
// 6 products, 2 squarings and one two-product sum.  All coordinates are Montgomery-form Fq, fully reduced.  All exceptional cases the
// reference's tests reach are handled: identity operands, P + P (doubling), P + (-P).
#pragma once
#include "field.cuh"

namespace pb200 {

struct alignas(16) G1Affine {
  Fq x, y;
};

struct alignas(16) G1XYZZ {
  Fq X, Y, ZZ, ZZZ;
  PB_HD bool is_inf() const { return ZZ.is_zero(); }
  static PB_HD G1XYZZ identity() {
    G1XYZZ r;
    r.X = Fq::zero(); r.Y = Fq::zero(); r.ZZ = Fq::zero(); r.ZZZ = Fq::zero();
    return r;
  }
};

PB_HD G1XYZZ g1_from_affine(const G1Affine& p) {
  G1XYZZ r;
  r.X = p.x; r.Y = p.y; r.ZZ = Fq::one(); r.ZZZ = Fq::one();
  return r;
}

// acc = 2 * (affine p)
PB_HD void g1_double_affine(G1XYZZ& acc, const G1Affine& p) {
  Fq U = fp_dbl(p.y);
  Fq V = fp_sqr(U);
  Fq W = fp_mul(U, V);
  Fq S = fp_mul(p.x, V);
  Fq M = fp_sqr(p.x);
  M = fp_add(fp_dbl(M), M);
  Fq X3 = fp_sub(fp_sqr(M), fp_dbl(S));
  acc.Y = fp_mul_sum2(M, fp_sub(S, X3), W, fp_neg(p.y));
  acc.X = X3;
  acc.ZZ = V;
  acc.ZZZ = W;
}

PB_HD void g1_double(G1XYZZ& a) {
  if (a.is_inf()) return;
  Fq U = fp_dbl(a.Y);
  Fq V = fp_sqr(U);
  Fq W = fp_mul(U, V);
  Fq S = fp_mul(a.X, V);
  Fq M = fp_sqr(a.X);
  M = fp_add(fp_dbl(M), M);
  Fq X3 = fp_sub(fp_sqr(M), fp_dbl(S));
  a.Y = fp_mul_sum2(M, fp_sub(S, X3), W, fp_neg(a.Y));
  a.X = X3;
  a.ZZ = fp_mul(V, a.ZZ);
  a.ZZZ = fp_mul(W, a.ZZZ);
}

// acc += p (p affine, never the identity)
PB_HD void g1_add_mixed(G1XYZZ& acc, const G1Affine& p) {
  if (acc.is_inf()) {
    acc = g1_from_affine(p);
    return;
  }
  Fq U2 = fp_mul(p.x, acc.ZZ);
  Fq S2 = fp_mul(p.y, acc.ZZZ);
  Fq Pd = fp_sub(U2, acc.X);
  Fq Rd = fp_sub(S2, acc.Y);
  if (Pd.is_zero()) {
    if (Rd.is_zero()) g1_double_affine(acc, p);
    else acc = G1XYZZ::identity();
    return;
  }
  Fq PP = fp_sqr(Pd);
  Fq PPP = fp_mul(Pd, PP);
  Fq Q = fp_mul(acc.X, PP);
  Fq X3 = fp_sub(fp_sub(fp_sqr(Rd), PPP), fp_dbl(Q));
  acc.Y = fp_mul_sum2(Rd, fp_sub(Q, X3), acc.Y, fp_neg(PPP));
  acc.X = X3;
  acc.ZZ = fp_mul(acc.ZZ, PP);
  acc.ZZZ = fp_mul(acc.ZZZ, PPP);
}

// acc += p with (almost) uniform control flow for SIMT execution: every lane runs the same 8M + 2S
// sequence; an empty accumulator is handled by a select at the end instead of an early return, and only
// the rare P == +-Q cases branch.
PB_HD void g1_add_mixed_uniform(G1XYZZ& acc, const G1Affine& p) {
  const bool was_inf = acc.is_inf();
  Fq U2 = fp_mul(p.x, acc.ZZ);
  Fq S2 = fp_mul(p.y, acc.ZZZ);
  Fq Pd = fp_sub(U2, acc.X);
  Fq Rd = fp_sub(S2, acc.Y);
  if (!was_inf && Pd.is_zero()) {
    if (Rd.is_zero()) g1_double_affine(acc, p);
    else acc = G1XYZZ::identity();
    return;
  }
  Fq PP = fp_sqr(Pd);
  Fq PPP = fp_mul(Pd, PP);
  Fq Q = fp_mul(acc.X, PP);
  Fq X3 = fp_sub(fp_sub(fp_sqr(Rd), PPP), fp_dbl(Q));
  Fq Y3 = fp_mul_sum2(Rd, fp_sub(Q, X3), acc.Y, fp_neg(PPP));
  Fq ZZ3 = fp_mul(acc.ZZ, PP);
  Fq ZZZ3 = fp_mul(acc.ZZZ, PPP);
  const Fq one = Fq::one();
#pragma unroll
  for (int i = 0; i < 8; i++) {
    acc.X.v[i] = was_inf ? p.x.v[i] : X3.v[i];
    acc.Y.v[i] = was_inf ? p.y.v[i] : Y3.v[i];
    acc.ZZ.v[i] = was_inf ? one.v[i] : ZZ3.v[i];
    acc.ZZZ.v[i] = was_inf ? one.v[i] : ZZZ3.v[i];
  }
}

// acc += q
PB_HD void g1_add(G1XYZZ& acc, const G1XYZZ& q) {
  if (q.is_inf()) return;
  if (acc.is_inf()) {
    acc = q;
    return;
  }
  Fq U1 = fp_mul(acc.X, q.ZZ);
  Fq U2 = fp_mul(q.X, acc.ZZ);
  Fq S1 = fp_mul(acc.Y, q.ZZZ);
  Fq S2 = fp_mul(q.Y, acc.ZZZ);
  Fq Pd = fp_sub(U2, U1);
  Fq Rd = fp_sub(S2, S1);
  if (Pd.is_zero()) {
    if (Rd.is_zero()) g1_double(acc);
    else acc = G1XYZZ::identity();
    return;
  }
  Fq PP = fp_sqr(Pd);
  Fq PPP = fp_mul(Pd, PP);
  Fq Q = fp_mul(U1, PP);
  Fq X3 = fp_sub(fp_sub(fp_sqr(Rd), PPP), fp_dbl(Q));
  acc.Y = fp_mul_sum2(Rd, fp_sub(Q, X3), S1, fp_neg(PPP));
  acc.X = X3;
  acc.ZZ = fp_mul(fp_mul(acc.ZZ, q.ZZ), PP);
  acc.ZZZ = fp_mul(fp_mul(acc.ZZZ, q.ZZZ), PPP);
}

// acc += q with select-based handling of identity operands (one instruction stream for all lanes, so two
// independent additions can be interleaved by the compiler); only the rare P == +-Q cases branch.
PB_HD void g1_add_uniform(G1XYZZ& acc, const G1XYZZ& q) {
  const bool a_inf = acc.is_inf(), q_inf = q.is_inf();
  Fq U1 = fp_mul(acc.X, q.ZZ);
  Fq U2 = fp_mul(q.X, acc.ZZ);
  Fq S1 = fp_mul(acc.Y, q.ZZZ);
  Fq S2 = fp_mul(q.Y, acc.ZZZ);
  Fq Pd = fp_sub(U2, U1);
  Fq Rd = fp_sub(S2, S1);
  if (!a_inf && !q_inf && Pd.is_zero()) {
    if (Rd.is_zero()) g1_double(acc);
    else acc = G1XYZZ::identity();
    return;
  }
  Fq PP = fp_sqr(Pd);
  Fq PPP = fp_mul(Pd, PP);
  Fq Q = fp_mul(U1, PP);
  Fq X3 = fp_sub(fp_sub(fp_sqr(Rd), PPP), fp_dbl(Q));
  Fq Y3 = fp_mul_sum2(Rd, fp_sub(Q, X3), S1, fp_neg(PPP));
  Fq ZZ3 = fp_mul(fp_mul(acc.ZZ, q.ZZ), PP);
  Fq ZZZ3 = fp_mul(fp_mul(acc.ZZZ, q.ZZZ), PPP);
#pragma unroll
  for (int i = 0; i < 8; i++) {
    acc.X.v[i] = q_inf ? acc.X.v[i] : (a_inf ? q.X.v[i] : X3.v[i]);
    acc.Y.v[i] = q_inf ? acc.Y.v[i] : (a_inf ? q.Y.v[i] : Y3.v[i]);
    acc.ZZ.v[i] = q_inf ? acc.ZZ.v[i] : (a_inf ? q.ZZ.v[i] : ZZ3.v[i]);
    acc.ZZZ.v[i] = q_inf ? acc.ZZZ.v[i] : (a_inf ? q.ZZZ.v[i] : ZZZ3.v[i]);
  }
}

PB_HD G1Affine g1_neg_affine(const G1Affine& p) {
  G1Affine r;
  r.x = p.x;
  r.y = fp_neg(p.y);
  return r;
}

// returns true when a is the identity (out untouched -> zeros)
PB_HD bool g1_to_affine(const G1XYZZ& a, G1Affine& out) {
  if (a.is_inf()) {
    out.x = Fq::zero();
    out.y = Fq::zero();
    return true;
  }
  Fq A = fp_inv(a.ZZZ);                  // 1/ZZZ
  Fq izz = fp_sqr(fp_mul(a.ZZ, A));      // (ZZ/ZZZ)^2 = 1/ZZ   (ZZ^3 == ZZZ^2)
  out.x = fp_mul(a.X, izz);
  out.y = fp_mul(a.Y, A);
  return false;
}

}  // namespace pb200
