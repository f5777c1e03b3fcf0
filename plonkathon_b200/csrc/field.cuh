// BN254 prime fields Fr (scalar field, curve.py:11 `field_modulus = b.curve_order`) and
// Fq (base field, py_ecc.bn128 `field_modulus`) for sm_100a.
//
// Replaces every py_ecc `FQ` operation the reference's hot path performs
// (`FQ.__add__/__sub__/__mul__/__truediv__/__pow__`, SURVEY App. A).
//
// Representation: 8 x u32 little-endian limbs, Montgomery form with R = 2^256 (the same
// encoding the .ptau SRS file uses on disk, setup.py:36-40), always fully reduced to [0, p).
// Both moduli are < 2^254, so a + b never overflows 256 bits.
//
// Montgomery product: operand-scanning CIOS split into an "even" and an "odd" accumulator so
// every 32x32->64 partial product lands on an aligned register pair; written as
// mad.lo.cc / madc.hi.cc pairs, which ptxas fuses into one IMAD.WIDE.U32.X each
// (136 IMAD-class instructions per product; checked with cuobjdump -sass).
// Squarings and the two-product sums of the group law (A B + C D) instead build the 512-bit product(s)
// with the same fused rows and reduce once (fp_sqr_wide / fp_mul_wide + fp_redc): 108 and 200
// multiplier instructions against 136 and 272.
//
// Every PTX instruction is wrapped in a tiny function that has a host emulation with an explicit
// carry flag, so the identical limb-level algorithm is unit-tested on the CPU
// (tests/test_host_arith.py via csrc/host_selftest.cpp) before it ever runs on a GPU.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PB_HD __host__ __device__ __forceinline__
#define PB_D __device__ __forceinline__
#else
#define PB_HD inline
#define PB_D inline
#endif

namespace pb200 {

// --------------------------------------------------------------------------------------------
// carry-chain primitives (device: PTX; host: emulation with an explicit flag)
// --------------------------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
PB_D uint32_t add_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t addc_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t addc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t sub_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t subc_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t subc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t mul_lo(uint32_t a, uint32_t b) { uint32_t r; asm volatile("mul.lo.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t mul_hi(uint32_t a, uint32_t b) { uint32_t r; asm volatile("mul.hi.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
PB_D uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm volatile("mad.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
PB_D uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm volatile("madc.lo.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
PB_D uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm volatile("madc.hi.cc.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
PB_D uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) { uint32_t r; asm volatile("madc.hi.u32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
#else
static thread_local uint32_t g_cf = 0;  // emulated CC.CF
inline uint32_t add_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b; g_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t addc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b + g_cf; g_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t addc(uint32_t a, uint32_t b) { return a + b + g_cf; }
inline uint32_t sub_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b; g_cf = (uint32_t)((t >> 32) & 1); return (uint32_t)t; }
inline uint32_t subc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b - g_cf; g_cf = (uint32_t)((t >> 32) & 1); return (uint32_t)t; }
inline uint32_t subc(uint32_t a, uint32_t b) { return a - b - g_cf; }
inline uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
inline uint32_t mul_hi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
inline uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (uint64_t)(uint32_t)(a * b) + c; g_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (uint64_t)(uint32_t)(a * b) + c + g_cf; g_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { uint64_t t = (((uint64_t)a * b) >> 32) + c + g_cf; g_cf = (uint32_t)(t >> 32); return (uint32_t)t; }
inline uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) { return (uint32_t)((((uint64_t)a * b) >> 32) + c + g_cf); }
#endif
// NB (device): borrow semantics of sub.cc/subc follow PTX: CC.CF holds the borrow-out and subc
// subtracts it; the host emulation mirrors that.

// --------------------------------------------------------------------------------------------
// field parameters
// --------------------------------------------------------------------------------------------
#define PB_LIMB_SWITCH(i, a0, a1, a2, a3, a4, a5, a6, a7) \
  ((i) == 0 ? a0 : (i) == 1 ? a1 : (i) == 2 ? a2 : (i) == 3 ? a3 : (i) == 4 ? a4 : (i) == 5 ? a5 : (i) == 6 ? a6 : a7)

struct FrParams {  // r = 21888242871839275222246405745257275088548364400416034343698204186575808495617
  static constexpr uint32_t NP0 = 0xefffffffu;  // -r^-1 mod 2^32
  static PB_HD constexpr uint32_t p(int i) { return PB_LIMB_SWITCH(i, 0xf0000001u, 0x43e1f593u, 0x79b97091u, 0x2833e848u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u); }
  static PB_HD constexpr uint32_t r1(int i) { return PB_LIMB_SWITCH(i, 0x4ffffffbu, 0xac96341cu, 0x9f60cd29u, 0x36fc7695u, 0x7879462eu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u); }
  static PB_HD constexpr uint32_t r2(int i) { return PB_LIMB_SWITCH(i, 0xae216da7u, 0x1bb8e645u, 0xe35c59e3u, 0x53fe3ab1u, 0x53bb8085u, 0x8c49833du, 0x7f4e44a5u, 0x0216d0b1u); }
  static PB_HD constexpr uint32_t r3(int i) { return PB_LIMB_SWITCH(i, 0xb4bf0040u, 0x5e94d8e1u, 0x1cfbb6b8u, 0x2a489cbeu, 0xa19fcfedu, 0x893cc664u, 0x7fcc657cu, 0x0cf8594bu); }
};

struct FqParams {  // q = 21888242871839275222246405745257275088696311157297823662689037894645226208583
  static constexpr uint32_t NP0 = 0xe4866389u;
  static PB_HD constexpr uint32_t p(int i) { return PB_LIMB_SWITCH(i, 0xd87cfd47u, 0x3c208c16u, 0x6871ca8du, 0x97816a91u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u); }
  static PB_HD constexpr uint32_t r1(int i) { return PB_LIMB_SWITCH(i, 0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u); }
  static PB_HD constexpr uint32_t r2(int i) { return PB_LIMB_SWITCH(i, 0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u, 0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u); }
  static PB_HD constexpr uint32_t r3(int i) { return PB_LIMB_SWITCH(i, 0xda1530dfu, 0xb1cd6dafu, 0xa7283db6u, 0x62f210e6u, 0x0ada0afbu, 0xef7f0b0cu, 0x2d592544u, 0x20fd6e90u); }
};

// --------------------------------------------------------------------------------------------
// field element
// --------------------------------------------------------------------------------------------
template <class P>
struct alignas(16) Fp {
  uint32_t v[8];

  static PB_HD Fp zero() { Fp r; for (int i = 0; i < 8; i++) r.v[i] = 0; return r; }
  static PB_HD Fp one() { Fp r; for (int i = 0; i < 8; i++) r.v[i] = P::r1(i); return r; }   // R mod p
  static PB_HD Fp r2() { Fp r; for (int i = 0; i < 8; i++) r.v[i] = P::r2(i); return r; }
  static PB_HD Fp r3() { Fp r; for (int i = 0; i < 8; i++) r.v[i] = P::r3(i); return r; }            // R^3 mod p
  static PB_HD Fp modulus() { Fp r; for (int i = 0; i < 8; i++) r.v[i] = P::p(i); return r; }

  PB_HD bool is_zero() const { uint32_t o = 0; for (int i = 0; i < 8; i++) o |= v[i]; return o == 0; }
  PB_HD bool operator==(const Fp& b) const { uint32_t o = 0; for (int i = 0; i < 8; i++) o |= v[i] ^ b.v[i]; return o == 0; }
  PB_HD bool operator!=(const Fp& b) const { return !(*this == b); }
};

// r = a - p if a >= p else a     (a < 2p < 2^256)
template <class P>
PB_HD void fp_reduce_once(Fp<P>& a) {
  uint32_t t[8];
  t[0] = sub_cc(a.v[0], P::p(0));
#pragma unroll
  for (int i = 1; i < 8; i++) t[i] = subc_cc(a.v[i], P::p(i));
  uint32_t borrow = subc(0u, 0u);  // 0xffffffff if a < p
#pragma unroll
  for (int i = 0; i < 8; i++) a.v[i] = borrow ? a.v[i] : t[i];
}

template <class P>
PB_HD Fp<P> fp_add(const Fp<P>& a, const Fp<P>& b) {
  Fp<P> r;
  r.v[0] = add_cc(a.v[0], b.v[0]);
#pragma unroll
  for (int i = 1; i < 7; i++) r.v[i] = addc_cc(a.v[i], b.v[i]);
  r.v[7] = addc(a.v[7], b.v[7]);
  fp_reduce_once(r);
  return r;
}

template <class P>
PB_HD Fp<P> fp_sub(const Fp<P>& a, const Fp<P>& b) {
  Fp<P> r;
  r.v[0] = sub_cc(a.v[0], b.v[0]);
#pragma unroll
  for (int i = 1; i < 8; i++) r.v[i] = subc_cc(a.v[i], b.v[i]);
  uint32_t mask = subc(0u, 0u);  // all ones if a < b
  r.v[0] = add_cc(r.v[0], P::p(0) & mask);
#pragma unroll
  for (int i = 1; i < 7; i++) r.v[i] = addc_cc(r.v[i], P::p(i) & mask);
  r.v[7] = addc(r.v[7], P::p(7) & mask);
  return r;
}

template <class P>
PB_HD Fp<P> fp_neg(const Fp<P>& a) {
  Fp<P> r;
  r.v[0] = sub_cc(P::p(0), a.v[0]);
#pragma unroll
  for (int i = 1; i < 7; i++) r.v[i] = subc_cc(P::p(i), a.v[i]);
  r.v[7] = subc(P::p(7), a.v[7]);
  uint32_t nz = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) nz |= a.v[i];
#pragma unroll
  for (int i = 0; i < 8; i++) r.v[i] = nz ? r.v[i] : 0u;
  return r;
}

template <class P>
PB_HD Fp<P> fp_dbl(const Fp<P>& a) { return fp_add(a, a); }

// ---- Montgomery product -------------------------------------------------------------------
// T = X + 2^32 * Y.  X holds the products of even limbs of the multiplicand, Y those of odd limbs,
// so each 64-bit partial product lands on the limb pair (2k, 2k+1) of its accumulator.
// acc(pairs 0..3) += a(0,2,4,6) * b, returns with CC.CF = carry out of limb 7
template <class P>
PB_HD void fp_mad_row(uint32_t* acc, const uint32_t* a, uint32_t b) {
  acc[0] = mad_lo_cc(a[0], b, acc[0]);
  acc[1] = madc_hi_cc(a[0], b, acc[1]);
#pragma unroll
  for (int j = 2; j < 8; j += 2) {
    acc[j] = madc_lo_cc(a[j], b, acc[j]);
    acc[j + 1] = madc_hi_cc(a[j], b, acc[j + 1]);
  }
}
// same with the modulus as multiplicand: acc += p(off, off+2, ..) * m
template <class P, int OFF>
PB_HD void fp_mad_row_mod(uint32_t* acc, uint32_t m) {
  acc[0] = mad_lo_cc(P::p(OFF), m, acc[0]);
  acc[1] = madc_hi_cc(P::p(OFF), m, acc[1]);
#pragma unroll
  for (int j = 2; j < 8; j += 2) {
    acc[j] = madc_lo_cc(P::p(OFF + j), m, acc[j]);
    acc[j + 1] = madc_hi_cc(P::p(OFF + j), m, acc[j + 1]);
  }
}

// One CIOS step.  State: T = U + 2^32 * V + w, where U is the 0-aligned accumulator, V the
// 32-bit-shifted one and w a pending 32-bit word of weight 1.
//   FIRST: U = a_even*b, V = a_odd*b, w = 0.
//   else : the previous step left (with roles swapped) an accumulator V whose low limb, together
//          with the previous w, sums to 0 mod 2^32.  Dividing T by 2^32 turns that accumulator into
//          (V >> 64) in the shifted role, its limb 1 becomes the new pending word, and the carry of
//          (low limb + old w), which is simply (old w != 0), enters the U row as carry-in.
// No 32-bit add ever touches half of a register pair, which keeps every row fusable into
// IMAD.WIDE.U32.X.
template <class P, bool FIRST>
PB_HD void fp_cios_step(uint32_t* U, uint32_t* V, uint32_t& w, const uint32_t* a, uint32_t b) {
  if (FIRST) {
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      U[j] = mul_lo(a[j], b);
      U[j + 1] = mul_hi(a[j], b);
      V[j] = mul_lo(a[j + 1], b);
      V[j + 1] = mul_hi(a[j + 1], b);
    }
    w = 0;
  } else {
    (void)add_cc(w, 0xffffffffu);  // CF = (w != 0)
    U[0] = madc_lo_cc(a[0], b, U[0]);
    U[1] = madc_hi_cc(a[0], b, U[1]);
#pragma unroll
    for (int j = 2; j < 8; j += 2) {
      U[j] = madc_lo_cc(a[j], b, U[j]);
      U[j + 1] = madc_hi_cc(a[j], b, U[j + 1]);
    }
    uint32_t c1 = addc(0u, 0u);  // carry out of U limb 7 == weight of V' limb 7
    w = V[1];
    V[0] = mad_lo_cc(a[1], b, V[2]);
    V[1] = madc_hi_cc(a[1], b, V[3]);
    V[2] = madc_lo_cc(a[3], b, V[4]);
    V[3] = madc_hi_cc(a[3], b, V[5]);
    V[4] = madc_lo_cc(a[5], b, V[6]);
    V[5] = madc_hi_cc(a[5], b, V[7]);
    V[6] = madc_lo_cc(a[7], b, 0u);
    V[7] = madc_hi(a[7], b, c1);
  }
  uint32_t m = mul_lo(U[0] + w, P::NP0);
  fp_mad_row_mod<P, 1>(V, m);
  fp_mad_row_mod<P, 0>(U, m);
  V[7] = addc(V[7], 0u);
}

#if !defined(__CUDA_ARCH__) && defined(PB_HOST_FAST_MUL)
// Host-only shortcut used by the library's own host code (final Horner / inversion of a commitment,
// transcript challenge reduction): 4 x 64-bit CIOS with unsigned __int128.  Same function value as the limb
// code below; the CPU unit tests build WITHOUT this macro so they exercise the device algorithm.
template <class P>
inline Fp<P> fp_mul_host64(const Fp<P>& a, const Fp<P>& b) {
  typedef unsigned __int128 u128;
  uint64_t A[4], B[4], M[4], T[6] = {0, 0, 0, 0, 0, 0};
  for (int i = 0; i < 4; i++) {
    A[i] = (uint64_t)a.v[2 * i] | ((uint64_t)a.v[2 * i + 1] << 32);
    B[i] = (uint64_t)b.v[2 * i] | ((uint64_t)b.v[2 * i + 1] << 32);
    M[i] = (uint64_t)P::p(2 * i) | ((uint64_t)P::p(2 * i + 1) << 32);
  }
  uint64_t np = 1;  // -p^-1 mod 2^64 by Newton iteration from the 32-bit constant's defining property
  for (int k = 0; k < 6; k++) np *= 2 - M[0] * np;
  np = (uint64_t)0 - np;
  for (int i = 0; i < 4; i++) {
    u128 c = 0;
    for (int j = 0; j < 4; j++) { c += (u128)A[j] * B[i] + T[j]; T[j] = (uint64_t)c; c >>= 64; }
    c += T[4]; T[4] = (uint64_t)c; T[5] = (uint64_t)(c >> 64);
    uint64_t m = T[0] * np;
    c = (u128)m * M[0] + T[0]; c >>= 64;
    for (int j = 1; j < 4; j++) { c += (u128)m * M[j] + T[j]; T[j - 1] = (uint64_t)c; c >>= 64; }
    c += T[4]; T[3] = (uint64_t)c; T[4] = T[5] + (uint64_t)(c >> 64); T[5] = 0;
  }
  // T < 2p: one conditional subtraction
  uint64_t r[4]; u128 br = 0; bool ge = T[4] != 0;
  if (!ge) { ge = true; for (int i = 3; i >= 0; i--) { if (T[i] != M[i]) { ge = T[i] > M[i]; break; } } }
  if (ge) { for (int i = 0; i < 4; i++) { u128 d = (u128)T[i] - M[i] - (uint64_t)br; r[i] = (uint64_t)d; br = (d >> 64) & 1; } }
  else { for (int i = 0; i < 4; i++) r[i] = T[i]; }
  Fp<P> o;
  for (int i = 0; i < 4; i++) { o.v[2 * i] = (uint32_t)r[i]; o.v[2 * i + 1] = (uint32_t)(r[i] >> 32); }
  return o;
}
#endif

template <class P>
PB_HD Fp<P> fp_mul(const Fp<P>& a, const Fp<P>& b) {
#if !defined(__CUDA_ARCH__) && defined(PB_HOST_FAST_MUL)
  return fp_mul_host64(a, b);
#else
  uint32_t X[8], Y[8], w;
  fp_cios_step<P, true>(X, Y, w, a.v, b.v[0]);
  fp_cios_step<P, false>(Y, X, w, a.v, b.v[1]);
  fp_cios_step<P, false>(X, Y, w, a.v, b.v[2]);
  fp_cios_step<P, false>(Y, X, w, a.v, b.v[3]);
  fp_cios_step<P, false>(X, Y, w, a.v, b.v[4]);
  fp_cios_step<P, false>(Y, X, w, a.v, b.v[5]);
  fp_cios_step<P, false>(X, Y, w, a.v, b.v[6]);
  fp_cios_step<P, false>(Y, X, w, a.v, b.v[7]);
  // last step had U = Y, V = X:  T / 2^32 = X + (Y >> 32) + (w != 0)
  Fp<P> r;
  (void)add_cc(w, 0xffffffffu);
  r.v[0] = addc_cc(X[0], Y[1]);
#pragma unroll
  for (int i = 1; i < 7; i++) r.v[i] = addc_cc(X[i], Y[i + 1]);
  r.v[7] = addc(X[7], 0u);
  fp_reduce_once(r);
  return r;
#endif
}

// ---- wide products and a separate Montgomery reduction ----------------------------------------------------------
// A 512-bit product is accumulated in two arrays: E holds the partial products that start at an even limb position
// (E[k] has weight 2^(32k)), O those that start at an odd one (O[k] has weight 2^(32(k+1))).  Every 64-bit partial
// product lands on an aligned pair (2k, 2k+1) of one array, so each row is a mad.lo.cc / madc.hi.cc chain that
// ptxas fuses into IMAD.WIDE.U32(.X), as in the CIOS product.  Unwritten limbs of E and O are zero.
//
// acc pairs (0,1) .. (2N-2,2N-1) += x[0] y, x[2] y, .., x[2N-2] y.
//   TOP  : acc[2N-1] is still zero and the row cannot carry out of it (the caller's bound on the partial sum).
//   else : the carry out of acc[2N-1] goes to acc[2N], which is still unwritten.
template <int N, bool TOP>
PB_HD void fp_wide_chain(uint32_t* acc, const uint32_t* x, uint32_t y) {
  acc[0] = mad_lo_cc(x[0], y, acc[0]);
#pragma unroll
  for (int k = 0; k < N; k++) {
    if (k > 0) acc[2 * k] = madc_lo_cc(x[2 * k], y, acc[2 * k]);
    if (TOP && k == N - 1) acc[2 * k + 1] = madc_hi(x[2 * k], y, 0u);
    else acc[2 * k + 1] = madc_hi_cc(x[2 * k], y, acc[2 * k + 1]);
  }
  if (!TOP) acc[2 * N] = addc(0u, 0u);
}

// E + 2^32 O = a * b (64 fused products).  Row i adds a * b_i at limb i; after row i the partial sum is below
// 2^(256 + 32 (i + 1)), which is what makes the TOP rows safe: their top limb is limb 8 + i.
PB_HD void fp_wide_rows(uint32_t* E, uint32_t* O, const uint32_t* a, const uint32_t* b) {
#pragma unroll
  for (int k = 0; k < 16; k++) { E[k] = 0; O[k] = 0; }
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    E[j] = mul_lo(a[j], b[0]);
    E[j + 1] = mul_hi(a[j], b[0]);
    O[j] = mul_lo(a[j + 1], b[0]);
    O[j + 1] = mul_hi(a[j + 1], b[0]);
  }
#pragma unroll
  for (int i = 1; i < 8; i++) {
    if (i & 1) {  // odd limbs of a land on even positions
      fp_wide_chain<4, true>(E + i + 1, a + 1, b[i]);
      fp_wide_chain<4, false>(O + i - 1, a, b[i]);
    } else {
      fp_wide_chain<4, false>(E + i, a, b[i]);
      fp_wide_chain<4, true>(O + i, a + 1, b[i]);
    }
  }
}

// T (16 limbs) = a * b
template <class P>
PB_HD void fp_mul_wide(uint32_t* T, const Fp<P>& a, const Fp<P>& b) {
  uint32_t E[16], O[16];
  fp_wide_rows(E, O, a.v, b.v);
  T[0] = E[0];
  T[1] = add_cc(E[1], O[0]);
#pragma unroll
  for (int k = 2; k < 15; k++) T[k] = addc_cc(E[k], O[k - 1]);
  T[15] = addc(E[15], O[14]);  // a * b < 2^512: no carry out
}

// T (16 limbs) += a * b; returns the carry out of limb 15 (the 17th limb of the sum)
template <class P>
PB_HD uint32_t fp_mad_wide(uint32_t* T, const Fp<P>& a, const Fp<P>& b) {
  uint32_t E[16], O[16];
  fp_wide_rows(E, O, a.v, b.v);
  T[0] = add_cc(T[0], E[0]);
#pragma unroll
  for (int k = 1; k < 15; k++) T[k] = addc_cc(T[k], E[k]);
  T[15] = addc_cc(T[15], E[15]);
  uint32_t c = addc(0u, 0u);
  T[1] = add_cc(T[1], O[0]);
#pragma unroll
  for (int k = 2; k < 16; k++) T[k] = addc_cc(T[k], O[k - 1]);
  return addc(c, 0u);
}

// T (16 limbs) = a^2: the 28 products a_i a_j (i < j) into E / O, doubled by a one-bit shift (their sum is below
// a^2 / 2 < 2^511), then the 8 squares a_i^2 on the pairs (2i, 2i+1): 36 fused products instead of 64.
template <class P>
PB_HD void fp_sqr_wide(uint32_t* T, const Fp<P>& a) {
  const uint32_t* x = a.v;
  uint32_t E[16], O[16];
#pragma unroll
  for (int k = 0; k < 16; k++) { E[k] = 0; O[k] = 0; }
  // row i: a_j a_i for j > i at position i + j; j - i odd -> O from index 2i, j - i even -> E from index 2i + 2
#pragma unroll
  for (int j = 1; j < 8; j += 2) {
    O[j - 1] = mul_lo(x[j], x[0]);
    O[j] = mul_hi(x[j], x[0]);
  }
#pragma unroll
  for (int j = 2; j < 8; j += 2) {
    E[j] = mul_lo(x[j], x[0]);
    E[j + 1] = mul_hi(x[j], x[0]);
  }
  fp_wide_chain<3, false>(O + 2, x + 2, x[1]);
  fp_wide_chain<3, true>(E + 4, x + 3, x[1]);
  fp_wide_chain<3, true>(O + 4, x + 3, x[2]);
  fp_wide_chain<2, false>(E + 6, x + 4, x[2]);
  fp_wide_chain<2, false>(O + 6, x + 4, x[3]);
  fp_wide_chain<2, true>(E + 8, x + 5, x[3]);
  fp_wide_chain<2, true>(O + 8, x + 5, x[4]);
  fp_wide_chain<1, false>(E + 10, x + 6, x[4]);
  fp_wide_chain<1, false>(O + 10, x + 6, x[5]);
  fp_wide_chain<1, true>(E + 12, x + 7, x[5]);
  fp_wide_chain<1, true>(O + 12, x + 7, x[6]);
  // D = E + 2^32 O (E[0] = E[1] = 0), then T = 2 D
  uint32_t D[16];
  D[0] = 0;
  D[1] = O[0];
  D[2] = add_cc(E[2], O[1]);
#pragma unroll
  for (int k = 3; k < 14; k++) D[k] = addc_cc(E[k], O[k - 1]);
  D[14] = addc_cc(O[13], 0u);
  D[15] = addc(0u, 0u);
#pragma unroll
  for (int k = 15; k > 0; k--) T[k] = (D[k] << 1) | (D[k - 1] >> 31);
  T[0] = mad_lo_cc(x[0], x[0], 0u);
  T[1] = madc_hi_cc(x[0], x[0], T[1]);
#pragma unroll
  for (int i = 1; i < 7; i++) {
    T[2 * i] = madc_lo_cc(x[i], x[i], T[2 * i]);
    T[2 * i + 1] = madc_hi_cc(x[i], x[i], T[2 * i + 1]);
  }
  T[14] = madc_lo_cc(x[7], x[7], T[14]);
  T[15] = madc_hi(x[7], x[7], T[15]);  // a^2 < 2^512: no carry out
}

// One word of the reduction, with the CIOS step's state T = U + 2^32 * V + w.  On entry V is the accumulator the
// previous step cleared (V[0] + w == 0 mod 2^32) and U the shifted one; dividing by 2^32 makes U aligned with
// carry-in (w != 0), the pending word becomes V[1] and V >> 64 takes the shifted role.  Then m clears U's low word.
//   FIRST: U = the low half of the input, V unused, w = 0.
// The state stays below 2^256 + 2^32 p < 2^288, so nothing carries out of the shifted accumulator's top limb.
template <class P, bool FIRST>
PB_HD void fp_redc_step(uint32_t* U, uint32_t* V, uint32_t& w) {
  uint32_t m;
  if (FIRST) {
    m = mul_lo(U[0], P::NP0);
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      V[j] = mul_lo(P::p(j + 1), m);
      V[j + 1] = mul_hi(P::p(j + 1), m);
    }
    fp_mad_row_mod<P, 0>(U, m);
    w = 0;
  } else {
    const uint32_t wn = V[1];
    (void)add_cc(w, 0xffffffffu);  // CF = (w != 0)
    m = mul_lo(addc(U[0], wn), P::NP0);
    V[0] = mad_lo_cc(P::p(1), m, V[2]);
    V[1] = madc_hi_cc(P::p(1), m, V[3]);
    V[2] = madc_lo_cc(P::p(3), m, V[4]);
    V[3] = madc_hi_cc(P::p(3), m, V[5]);
    V[4] = madc_lo_cc(P::p(5), m, V[6]);
    V[5] = madc_hi_cc(P::p(5), m, V[7]);
    V[6] = madc_lo_cc(P::p(7), m, 0u);
    V[7] = madc_hi(P::p(7), m, 0u);
    (void)add_cc(w, 0xffffffffu);
    U[0] = madc_lo_cc(P::p(0), m, U[0]);
    U[1] = madc_hi_cc(P::p(0), m, U[1]);
#pragma unroll
    for (int j = 2; j < 8; j += 2) {
      U[j] = madc_lo_cc(P::p(j), m, U[j]);
      U[j + 1] = madc_hi_cc(P::p(j), m, U[j + 1]);
    }
    w = wn;
  }
  V[7] = addc(V[7], 0u);  // carry out of U limb 7
}

// Montgomery reduction T R^-1 mod p of a 16-limb T < p 2^256, fully reduced.  The eight steps reduce the low half
// to (T_lo + m p) / 2^256 <= p (m < 2^256); the high half T_hi < p is added after, and the sum is below 2p.
// 72 multiplier instructions: 8 for the words m, 64 fused for m p.
template <class P>
PB_HD Fp<P> fp_redc(const uint32_t* T) {
  uint32_t X[8], Y[8], w;
#pragma unroll
  for (int i = 0; i < 8; i++) X[i] = T[i];
  fp_redc_step<P, true>(X, Y, w);
  fp_redc_step<P, false>(Y, X, w);
  fp_redc_step<P, false>(X, Y, w);
  fp_redc_step<P, false>(Y, X, w);
  fp_redc_step<P, false>(X, Y, w);
  fp_redc_step<P, false>(Y, X, w);
  fp_redc_step<P, false>(X, Y, w);
  fp_redc_step<P, false>(Y, X, w);
  // last step had U = Y, V = X:  (T_lo + m p) / 2^256 = X + (Y >> 32) + (w != 0)
  Fp<P> r;
  (void)add_cc(w, 0xffffffffu);
  r.v[0] = addc_cc(X[0], Y[1]);
#pragma unroll
  for (int i = 1; i < 7; i++) r.v[i] = addc_cc(X[i], Y[i + 1]);
  r.v[7] = addc(X[7], 0u);
  r.v[0] = add_cc(r.v[0], T[8]);
#pragma unroll
  for (int i = 1; i < 7; i++) r.v[i] = addc_cc(r.v[i], T[8 + i]);
  r.v[7] = addc(r.v[7], T[15]);
  fp_reduce_once(r);
  return r;
}

// a^2 R^-1 mod p: 108 multiplier instructions instead of the product's 136
template <class P>
PB_HD Fp<P> fp_sqr(const Fp<P>& a) {
#if !defined(__CUDA_ARCH__) && defined(PB_HOST_FAST_MUL)
  return fp_mul_host64(a, a);
#else
  uint32_t T[16];
  fp_sqr_wide(T, a);
  return fp_redc<P>(T);
#endif
}

// (a b + c d) R^-1 mod p with one reduction, for the A B - C D shape of the group law (pass C and p - D).
// a, b, c, d < p, so a b + c d < 2 p^2 < p 2^256 because 2p < 2^256: the reduction's input bound holds and the
// 512-bit sum does not carry out.  200 multiplier instructions instead of two products' 272.
template <class P>
PB_HD Fp<P> fp_mul_sum2(const Fp<P>& a, const Fp<P>& b, const Fp<P>& c, const Fp<P>& d) {
#if !defined(__CUDA_ARCH__) && defined(PB_HOST_FAST_MUL)
  return fp_add(fp_mul_host64(a, b), fp_mul_host64(c, d));
#else
  uint32_t T[16];
  fp_mul_wide(T, a, b);
  (void)fp_mad_wide(T, c, d);
  return fp_redc<P>(T);
#endif
}

template <class P>
PB_HD Fp<P> fp_to_mont(const Fp<P>& a) { return fp_mul(a, Fp<P>::r2()); }

// to_mont for an arbitrary 256-bit input (not necessarily < p): CIOS only needs one operand below p
template <class P>
PB_HD Fp<P> fp_to_mont_any(const Fp<P>& a) { return fp_mul(Fp<P>::r2(), a); }

template <class P>
PB_HD Fp<P> fp_from_mont(const Fp<P>& a) {
  Fp<P> o = Fp<P>::zero();
  o.v[0] = 1;
  return fp_mul(a, o);
}

// a^e for a 256-bit exponent given as 8 LE limbs (vartime in e; e is public everywhere it is used)
template <class P>
PB_HD Fp<P> fp_pow(const Fp<P>& a, const uint32_t* e) {
  Fp<P> r = Fp<P>::one();
  bool started = false;
  for (int i = 255; i >= 0; i--) {
    if (started) r = fp_sqr(r);
    if ((e[i >> 5] >> (i & 31)) & 1) {
      r = started ? fp_mul(r, a) : a;
      started = true;
    }
  }
  return r;
}

template <class P>
PB_HD Fp<P> fp_pow_u64(const Fp<P>& a, uint64_t e) {
  uint32_t ee[8] = {(uint32_t)e, (uint32_t)(e >> 32), 0, 0, 0, 0, 0, 0};
  return fp_pow(a, ee);
}

// inverse by Fermat (a^(p-2)); inv(0) == 0, matching py_ecc's prime_field_inv convention
template <class P>
PB_HD Fp<P> fp_inv(const Fp<P>& a) {
  uint32_t e[8];
#pragma unroll
  for (int i = 0; i < 8; i++) e[i] = P::p(i);
  e[0] -= 2;  // p is odd and p(0) >= 2 for both fields
  return fp_pow(a, e);
}

typedef Fp<FrParams> Fr;
typedef Fp<FqParams> Fq;

}  // namespace pb200
