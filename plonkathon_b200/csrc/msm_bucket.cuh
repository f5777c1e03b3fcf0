// Bucket reduction of the G1 MSM (msm.cu) and the batched-affine alternative for its bucket accumulation: the
// thread bodies.
//
// Replaces the additions of curve.py:38-111 (`ec_lincomb` over py_ecc `add`, one field inversion per addition).
//
// Accumulation, `PB200_MSM_ACC=affine` only (the default is the XYZZ segment kernel in msm.cu; this one is exact
// but measured slower on B200, profiles/r02_msm_affine_vs_xyzz.md) = rounds of pairwise AFFINE additions that share
// one inversion per thread (Montgomery's trick):
// 6 field products per addition (1 forward, 5 backward) instead of 10 for an XYZZ += affine step, plus one
// safegcd inversion (modinv.cuh, no multiplication chain) amortised over the B additions of a thread.
//
// Layout.  The counting sort (msm.cu) leaves the entries of bucket b -- point index | sign << 31 -- at positions
// [off[b], off[b] + cnt[b]) of `sorted`, with every off[b] EVEN (counts are padded to even for the scan; the pad
// position holds PB_MSM_PAD).  Slot s of the point array `pts` stands for positions 2s and 2s+1, so bucket b
// owns slots [off[b]/2, off[b]/2 + m0), m0 = ceil(cnt[b] / 2).
//   round 0   : slot s <- table[sorted[2s]] + table[sorted[2s+1]], or a plain copy when 2s+1 is the pad.
//               Dense (every slot has work): a warp owns 32*B consecutive slots, lane-interleaved (coalesced).
//   round r>=1: in place, within each bucket: slot base + 2^r j  +=  slot base + 2^r j + 2^(r-1)  whenever the
//               right-hand slot is below m0.  Thread t owns the slot range [t B 2^r, (t+1) B 2^r) and walks the
//               buckets that intersect it (at most B additions).  A right-hand slot is never the left-hand slot
//               of another addition of the same round, so rounds need no synchronisation inside a launch.
// After ceil(log2(max cnt)) rounds slot off[b]/2 holds the sum of bucket b.  Rounds whose stride exceeds every
// bucket return at once (device-side max count), so no host round trip decides the round count.
// Exceptional cases are exact, as the reference's group law has them: equal points are doubled (tangent slope,
// denominator 2y), opposite points give the identity (encoded x.v[7] == 0xffffffff, not a reduced element), an
// identity operand returns the other one.
//
// Reduction = sum_j (j+1) B_j by recursive grouping: level 0 turns g consecutive buckets into
// (S, R) = (sum B, sum (lo+1) B) with one thread per group (running sums, all the work, full width); with
// F = G sum_i i S_i + sum_i R_i as the invariant (G = product of the group sizes below), a higher level folds 1024
// elements into S' = sum S, R' = G sum_lo lo S_lo + sum R with one block per group (suffix scan + tree).
//
// The bodies are host/device functions so tests/test_host_arith.py can run the whole pipeline on the CPU
// (csrc/host_selftest.cpp) against the oracle's group law; the __global__ wrappers live in msm.cu.
#pragma once
#include "curve.cuh"
#include "modinv.cuh"
#if !defined(__CUDA_ARCH__)
#include <stdio.h>
#include <stdlib.h>
#endif

namespace pb200 {

#define PB_AFF_ADD 1u
#define PB_AFF_DBL 2u
#define PB_AFF_INDEX_BITS 29
#define PB_AFF_INDEX_MASK ((1u << PB_AFF_INDEX_BITS) - 1)
#define PB_AFF_BMAX 128         // capacity of a thread's chain of additions (one inversion per chain)
#define PB_MSM_PAD 0xffffffffu  // `sorted` filler of padding positions
#define PB_AFF_GRID_ROUNDS 12   // rounds launched grid-wide (buckets up to 4096 entries); the rest: one-block tail

struct AffAcc {
  const G1Affine* table;    // point table (Montgomery affine), addressed through `sorted`
  const uint32_t* sorted;   // 2 * S entries
  G1Affine* pts;            // S slots
  const uint32_t* off;      // nbl + 1 even offsets (entry positions)
  const uint32_t* cnt;      // nbl bucket sizes
  const uint32_t* max_cnt;  // largest bucket size (device scalar)
  uint32_t nbl;             // buckets of this launch (all bucket sets)
  uint32_t r;               // round
  uint32_t B;               // round 0: slots (= additions) per thread; round r >= 1: a thread's range is B * 2^(r-1)
                            // slots, which holds at most B additions (left-hand slots are more than 2^(r-1) apart)
                            // and about B / 2 when the buckets are large.  B <= PB_AFF_BMAX.
};

PB_HD bool aff_is_identity_x(const Fq& x) { return x.v[7] == 0xffffffffu; }
PB_HD G1Affine aff_identity() {
  G1Affine r;
  for (int i = 0; i < 8; i++) { r.x.v[i] = 0xffffffffu; r.y.v[i] = 0; }
  return r;
}

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ Fq aff_ld_fq(const Fq* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = __ldg(q), b = __ldg(q + 1);
  Fq r;
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
// plain (coherent) loads for the in-place point array, which the same launch also writes
__device__ __forceinline__ Fq aff_ld_fq_rw(const Fq* p) {
  const uint4* q = reinterpret_cast<const uint4*>(p);
  uint4 a = q[0], b = q[1];
  Fq r;
  r.v[0] = a.x; r.v[1] = a.y; r.v[2] = a.z; r.v[3] = a.w;
  r.v[4] = b.x; r.v[5] = b.y; r.v[6] = b.z; r.v[7] = b.w;
  return r;
}
__device__ __forceinline__ void aff_st_fq(Fq* p, const Fq& r) {
  uint4* q = reinterpret_cast<uint4*>(p);
  q[0] = make_uint4(r.v[0], r.v[1], r.v[2], r.v[3]);
  q[1] = make_uint4(r.v[4], r.v[5], r.v[6], r.v[7]);
}
__device__ __forceinline__ uint32_t aff_ld_u32(const uint32_t* p) { return __ldg(p); }
#else
inline Fq aff_ld_fq(const Fq* p) { return *p; }
inline Fq aff_ld_fq_rw(const Fq* p) { return *p; }
inline void aff_st_fq(Fq* p, const Fq& r) { *p = r; }
inline uint32_t aff_ld_u32(const uint32_t* p) { return *p; }
#endif

PB_HD void aff_st_point(G1Affine* dst, const G1Affine& p) {
  aff_st_fq(&dst->x, p.x);
  aff_st_fq(&dst->y, p.y);
}
// table point of a sorted entry, sign applied
PB_HD Fq aff_entry_x(const AffAcc& a, uint32_t e) { return aff_ld_fq(&a.table[e & 0x7fffffffu].x); }
PB_HD Fq aff_entry_y(const AffAcc& a, uint32_t e) {
  Fq y = aff_ld_fq(&a.table[e & 0x7fffffffu].y);
  return (e >> 31) ? fp_neg(y) : y;
}

// first index i in [lo, hi) with a[i] > key (hi if none)
PB_HD uint32_t aff_upper_bound(const uint32_t* a, uint32_t lo, uint32_t hi, uint32_t key) {
  while (lo < hi) {
    uint32_t mid = (lo + hi) >> 1;
    if (aff_ld_u32(a + mid) > key) hi = mid; else lo = mid + 1;
  }
  return lo;
}

// the shared tail of an addition: p + q (kind ADD) or 2p (kind DBL) given 1/d
PB_HD G1Affine aff_finish(const G1Affine& p, const G1Affine& q, uint32_t kind, const Fq& dinv) {
  Fq num;
  if (kind == PB_AFF_ADD) {
    num = fp_sub(q.y, p.y);
  } else {
    Fq xx = fp_sqr(p.x);
    num = fp_add(fp_dbl(xx), xx);
  }
  const Fq lam = fp_mul(num, dinv);
  G1Affine r;
  r.x = fp_sub(fp_sub(fp_sqr(lam), p.x), q.x);
  r.y = fp_sub(fp_mul(lam, fp_sub(p.x, r.x)), p.y);
  return r;
}

// classify the pair (x1 == x2 case): returns the denominator and kind, or kind 0 for P + (-P)
PB_HD uint32_t aff_classify_equal_x(const Fq& y1, const Fq& y2, Fq& d) {
  if (y1 == y2) {  // y != 0: the group has odd order
    d = fp_dbl(y1);
    return PB_AFF_DBL;
  }
  return 0;
}

// slots per thread in round r
PB_HD uint64_t aff_round_span(uint32_t B, uint32_t r) { return r == 0 ? B : (uint64_t)B << (r - 1); }
// threads a grid-wide launch of round r needs for S_bound slots
PB_HD uint64_t aff_round_threads(uint64_t s_bound, uint32_t B, uint32_t r) {
  const uint64_t per = aff_round_span(B, r);
  uint64_t t = (s_bound + per - 1) / per;
  return r == 0 ? ((t + 31) / 32) * 32 : t;  // round 0 hands whole warps 32 * B slots
}

// ---- round 0 of thread t: table -> pts ----------------------------------------------------------------------
PB_HD void aff_round0_thread(const AffAcc& a, uint64_t t, Fq* pref, uint32_t* desc) {
  const uint32_t S = aff_ld_u32(a.off + a.nbl) >> 1;
  const uint64_t w0 = (t >> 5) * 32ull * a.B;
  if (w0 >= S) return;
  const uint32_t w1 = (uint32_t)(w0 + 32ull * a.B < S ? w0 + 32ull * a.B : S);
  Fq acc = Fq::one();
  uint32_t K = 0;
  for (uint32_t s = (uint32_t)w0 + (uint32_t)(t & 31); s < w1; s += 32) {
    const uint32_t e0 = aff_ld_u32(a.sorted + 2 * s), e1 = aff_ld_u32(a.sorted + 2 * s + 1);
    if (e1 == PB_MSM_PAD) {  // the bucket's odd last entry: carried over
      G1Affine p;
      p.x = aff_entry_x(a, e0);
      p.y = aff_entry_y(a, e0);
      aff_st_point(a.pts + s, p);
      continue;
    }
    const Fq x1 = aff_entry_x(a, e0), x2 = aff_entry_x(a, e1);
    Fq d = fp_sub(x2, x1);
    uint32_t kind = PB_AFF_ADD;
    if (d.is_zero()) {
      kind = aff_classify_equal_x(aff_entry_y(a, e0), aff_entry_y(a, e1), d);
      if (kind == 0) {
        aff_st_point(a.pts + s, aff_identity());
        continue;
      }
    }
    pref[K] = acc;
    desc[K] = s | (kind << PB_AFF_INDEX_BITS);
    K++;
    acc = fp_mul(acc, d);
  }
  Fq inv = fp_inv_gcd(acc);
  while (K > 0) {
    K--;
    const uint32_t s = desc[K] & PB_AFF_INDEX_MASK, kind = desc[K] >> PB_AFF_INDEX_BITS;
    const uint32_t e0 = aff_ld_u32(a.sorted + 2 * s), e1 = aff_ld_u32(a.sorted + 2 * s + 1);
    G1Affine p, q;
    p.x = aff_entry_x(a, e0); p.y = aff_entry_y(a, e0);
    q.x = aff_entry_x(a, e1); q.y = aff_entry_y(a, e1);
    const Fq d = kind == PB_AFF_ADD ? fp_sub(q.x, p.x) : fp_dbl(p.y);
    const Fq dinv = fp_mul(inv, pref[K]);
    inv = fp_mul(inv, d);
    aff_st_point(a.pts + s, aff_finish(p, q, kind, dinv));
  }
}

// ---- round r >= 1 of thread t: in place on pts ----------------------------------------------------------------
PB_HD void aff_round_thread(const AffAcc& a, uint64_t t, Fq* pref, uint32_t* desc) {
  const uint32_t r = a.r;
  if (r >= 32 || aff_ld_u32(a.max_cnt) <= (1u << r)) return;  // every bucket has m0 <= 2^(r-1): nothing to pair
  const uint32_t S = aff_ld_u32(a.off + a.nbl) >> 1;
  const uint64_t step = 1ull << r, hs = step >> 1;
  const uint64_t span = a.B * hs;  // two left-hand slots are at least hs + 1 apart: at most B of them in the range
  const uint64_t lo64 = t * span;
  if (lo64 >= S) return;
  const uint32_t lo = (uint32_t)lo64;
  const uint32_t hi = (uint32_t)(lo64 + span < S ? lo64 + span : S);
  uint32_t b = aff_upper_bound(a.off, 0, a.nbl + 1, 2 * lo) - 1;  // off[b] <= 2 lo < off[b+1]
  Fq acc = Fq::one();
  uint32_t K = 0;
  for (; b < a.nbl; b++) {
    const uint32_t base = aff_ld_u32(a.off + b) >> 1;
    if (base >= hi) break;
    const uint32_t m0 = (aff_ld_u32(a.cnt + b) + 1) >> 1;
    if (m0 <= hs) continue;
    uint64_t u = lo > base ? (((uint64_t)(lo - base) + step - 1) >> r) << r : 0;
    for (; base + u < hi && u + hs < m0; u += step) {
      const uint32_t left = base + (uint32_t)u, right = left + (uint32_t)hs;
      const Fq x1 = aff_ld_fq_rw(&a.pts[left].x), x2 = aff_ld_fq_rw(&a.pts[right].x);
      if (aff_is_identity_x(x2)) continue;  // P + 0
      if (aff_is_identity_x(x1)) {          // 0 + Q
        G1Affine q;
        q.x = x2;
        q.y = aff_ld_fq_rw(&a.pts[right].y);
        aff_st_point(a.pts + left, q);
        continue;
      }
      Fq d = fp_sub(x2, x1);
      uint32_t kind = PB_AFF_ADD;
      if (d.is_zero()) {
        kind = aff_classify_equal_x(aff_ld_fq_rw(&a.pts[left].y), aff_ld_fq_rw(&a.pts[right].y), d);
        if (kind == 0) {
          aff_st_point(a.pts + left, aff_identity());
          continue;
        }
      }
#if !defined(__CUDA_ARCH__)
      if (K >= a.B) { fprintf(stderr, "aff_round_thread: chain longer than B\n"); abort(); }  // host self-test only
#endif
      pref[K] = acc;
      desc[K] = left | (kind << PB_AFF_INDEX_BITS);
      K++;
      acc = fp_mul(acc, d);
    }
  }
  Fq inv = fp_inv_gcd(acc);
  while (K > 0) {
    K--;
    const uint32_t left = desc[K] & PB_AFF_INDEX_MASK, kind = desc[K] >> PB_AFF_INDEX_BITS;
    const uint32_t right = left + (uint32_t)hs;
    G1Affine p, q;
    p.x = aff_ld_fq_rw(&a.pts[left].x); p.y = aff_ld_fq_rw(&a.pts[left].y);
    q.x = aff_ld_fq_rw(&a.pts[right].x); q.y = aff_ld_fq_rw(&a.pts[right].y);
    const Fq d = kind == PB_AFF_ADD ? fp_sub(q.x, p.x) : fp_dbl(p.y);
    const Fq dinv = fp_mul(inv, pref[K]);
    inv = fp_mul(inv, d);
    aff_st_point(a.pts + left, aff_finish(p, q, kind, dinv));
  }
}

// ---- bucket reduction -----------------------------------------------------------------------------------------
struct SR {
  G1XYZZ S, R;
};

// acc += p when take (select-based: one instruction stream for all lanes; only P == +-Q branches)
PB_HD void g1_add_mixed_sel(G1XYZZ& acc, const G1Affine& p, bool take) {
  const bool was_inf = acc.is_inf();
  Fq U2 = fp_mul(p.x, acc.ZZ);
  Fq S2 = fp_mul(p.y, acc.ZZZ);
  Fq Pd = fp_sub(U2, acc.X);
  Fq Rd = fp_sub(S2, acc.Y);
  if (take && !was_inf && Pd.is_zero()) {
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
    acc.X.v[i] = !take ? acc.X.v[i] : (was_inf ? p.x.v[i] : X3.v[i]);
    acc.Y.v[i] = !take ? acc.Y.v[i] : (was_inf ? p.y.v[i] : Y3.v[i]);
    acc.ZZ.v[i] = !take ? acc.ZZ.v[i] : (was_inf ? one.v[i] : ZZ3.v[i]);
    acc.ZZZ.v[i] = !take ? acc.ZZZ.v[i] : (was_inf ? one.v[i] : ZZZ3.v[i]);
  }
}

struct ReduceArgs {
  // level 0 input: bucket sums in the slot array
  const G1Affine* pts;
  const uint32_t* off;
  const uint32_t* cnt;
  const G1XYZZ* xb;   // alternative level 0 input: one XYZZ point per bucket (nullptr: use pts / off / cnt)
  SR* out;
  uint32_t sets;      // bucket sets (windows / batched commitments)
  uint32_t m;         // buckets per set
  uint32_t g;         // group size
};
PB_HD uint32_t reduce_groups(uint32_t m, uint32_t g) { return (m + g - 1) / g; }

// acc += bucket b (level-0 input: the slot array of the affine accumulation, or XYZZ buckets when a.xb is set)
PB_HD void reduce_level0_fetch(const ReduceArgs& a, uint32_t b, G1XYZZ& acc) {
  if (a.xb) {
    const G1XYZZ v = a.xb[b];
    g1_add_uniform(acc, v);
    return;
  }
  const bool live = aff_ld_u32(a.cnt + b) != 0;
  const uint32_t slot = live ? aff_ld_u32(a.off + b) >> 1 : 0;
  G1Affine p;
  p.x = aff_ld_fq(&a.pts[slot].x);
  p.y = aff_ld_fq(&a.pts[slot].y);
  g1_add_mixed_sel(acc, p, live && !aff_is_identity_x(p.x));
}

// level 0, thread t = set * groups + gi: (S, R) = (sum B_j, sum (lo + 1) B_j) over the group's buckets
PB_HD void reduce_level0_thread(const ReduceArgs& a, uint64_t t) {
  const uint32_t groups = reduce_groups(a.m, a.g);
  if (t >= (uint64_t)a.sets * groups) return;
  const uint32_t set = (uint32_t)(t / groups), gi = (uint32_t)(t % groups);
  const uint32_t j0 = gi * a.g;
  const uint32_t len = a.m - j0 < a.g ? a.m - j0 : a.g;
  const uint32_t b0 = set * a.m + j0;
  // running sums from the top: acc_k = B_k + acc_(k+1), sum = sum_k acc_k.  sum += acc_k and acc_(k-1) = acc_k + B_(k-1)
  // do not depend on each other, so the two additions of an iteration can be interleaved
  G1XYZZ acc = G1XYZZ::identity(), sum = G1XYZZ::identity();
  reduce_level0_fetch(a, b0 + len - 1, acc);
  for (uint32_t k = len; k-- > 0;) {
    G1XYZZ nxt = acc;
    if (k > 0) reduce_level0_fetch(a, b0 + k - 1, nxt);
    g1_add_uniform(sum, acc);
    acc = nxt;
  }
  SR o;
  o.S = acc;
  o.R = sum;
  a.out[t] = o;
}

// ---- levels >= 1: one block of 128 threads folds a chunk of 512 elements --------------------------------------
// Above level 0 there are too few elements to fill the machine, so a level is bound by the length of its chains of
// dependent additions, not by throughput: a block-wide suffix scan and a tree keep that length at ~23 additions for
// a group of 512 (a thread-per-group level of 16 has 48, and more than twice as many levels).
//   element index in the chunk: lo = 4 t + e, e < 4;   S' = sum S,   R' = G sum_lo lo S_lo + sum R
//   thread t: s_t = sum_e S, w_t = sum_e e S_e, r_t = sum_e R  ->  x_t = r_t + G w_t
//   suffix scan: suf_t = sum_{t' >= t} s_t'                     ->  S' = suf_0, sum_t t s_t = sum_{t >= 1} suf_t
//   y_t = x_t + 4 G suf_t (t >= 1), tree sum of y               ->  R'
// One out-of-line copy of the two group operations for the block-wide levels: inlined at every use they made
// k_reduce_block ~50k instructions of straight-line code that each block runs once -- an instruction-cache miss on
// every line (measured: 11 us per addition instead of ~5).
#if defined(__CUDA_ARCH__)
static __device__ __noinline__ void blk_add(G1XYZZ& acc, const G1XYZZ& q) { g1_add(acc, q); }
static __device__ __noinline__ void blk_double(G1XYZZ& a) { g1_double(a); }
#else
inline void blk_add(G1XYZZ& acc, const G1XYZZ& q) { g1_add(acc, q); }
inline void blk_double(G1XYZZ& a) { g1_double(a); }
#endif

// 128 threads = one warp per SM sub-partition: the integer pipe of a sub-partition serves one dependent chain at
// full speed, two warps on it would each run their chain at half speed (measured: 256-thread blocks took ~10 us per
// addition, twice the single-warp latency)
#define PB_REDUCE_THREADS 128
#define PB_REDUCE_CHUNK (4 * PB_REDUCE_THREADS)
struct BlockLevelArgs {
  const SR* in;
  SR* out;
  uint32_t sets, m;   // input elements per set
  uint32_t log_G;     // log2 of the weight G of this level's element index
};
PB_HD uint32_t reduce_chunks(uint32_t m) { return (m + PB_REDUCE_CHUNK - 1) / PB_REDUCE_CHUNK; }

PB_HD void blk_local(const BlockLevelArgs& a, uint32_t set, uint32_t chunk, uint32_t t, G1XYZZ& s, G1XYZZ& x) {
  const uint64_t i0 = (uint64_t)chunk * PB_REDUCE_CHUNK + 4 * t;
  const SR* base = a.in + (uint64_t)set * a.m;
  G1XYZZ acc = G1XYZZ::identity(), w = G1XYZZ::identity(), r = G1XYZZ::identity();
#pragma unroll 1
  for (int e = 3; e >= 0; e--) {
    if (i0 + e >= a.m) continue;
    const SR v = base[i0 + e];
    blk_add(acc, v.S);
    if (e >= 1) blk_add(w, acc);
    blk_add(r, v.R);
  }
#pragma unroll 1
  for (uint32_t d = 0; d < a.log_G; d++) blk_double(w);
  blk_add(r, w);
  s = acc;
  x = r;
}
// one Hillis-Steele step of the inclusive suffix scan: value of position t after combining with t + d
PB_HD G1XYZZ blk_scan_step(const G1XYZZ* sh, uint32_t t, uint32_t d) {
  G1XYZZ v = sh[t];
  if (t + d < PB_REDUCE_THREADS) {
    const G1XYZZ o = sh[t + d];
    blk_add(v, o);
  }
  return v;
}
PB_HD G1XYZZ blk_weight(const BlockLevelArgs& a, uint32_t t, const G1XYZZ& x, G1XYZZ suf) {
  G1XYZZ y = x;
  if (t >= 1) {
#pragma unroll 1
    for (uint32_t d = 0; d < a.log_G + 2; d++) blk_double(suf);
    blk_add(y, suf);
  }
  return y;
}
PB_HD void blk_tree_step(G1XYZZ* sh, uint32_t t, uint32_t d) {
  if (t < d) {
    G1XYZZ u = sh[t];
    const G1XYZZ v = sh[t + d];
    blk_add(u, v);
    sh[t] = u;
  }
}

// the last few elements of a set (host code in msm.cu): (S, R) <- (sum S, G sum_i i S_i + sum R)
PB_HD SR reduce_fold_final(const SR* e, uint32_t count, uint32_t log_G) {
  G1XYZZ acc = G1XYZZ::identity(), w = G1XYZZ::identity(), r = G1XYZZ::identity();
  for (uint32_t k = count; k-- > 0;) {
    g1_add(acc, e[k].S);
    if (k >= 1) g1_add(w, acc);
    g1_add(r, e[k].R);
  }
  for (uint32_t d = 0; d < log_G; d++) g1_double(w);
  g1_add(r, w);
  SR o;
  o.S = acc;
  o.R = r;
  return o;
}

}  // namespace pb200
