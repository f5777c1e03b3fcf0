// Host build of the limb-level arithmetic in field.cuh / curve.cuh (same code path as the device,
// PTX carry-chain primitives replaced by their emulation).  TEST INFRASTRUCTURE: loaded only by
// tests/test_host_arith.py and tests/test_field_wide.py through ctypes; never linked into libplonk_b200.so.
#include "field.cuh"
#include "curve.cuh"
#include "msm_digits.cuh"
#include "modinv.cuh"
#include "msm_bucket.cuh"
#include "ntt_shard.cuh"
#include <vector>
#include <cstring>
using namespace pb200;

template <class F> static F ld(const uint32_t* p) { F r; memcpy(r.v, p, 32); return r; }
template <class F> static void st(uint32_t* p, const F& a) { memcpy(p, a.v, 32); }

extern "C" {
// op: 0 add, 1 sub, 2 mul, 3 neg, 4 inv, 5 to_mont, 6 from_mont, 7 dbl, 8 sqr, 9 inv by safegcd (Montgomery
// contract of op 4), 10 plain-integer inverse by safegcd ; field: 0 Fr, 1 Fq
int hs_field_op(int field, int op, const uint32_t* a, const uint32_t* b, uint32_t* out) {
#define RUN(F)                                                   \
  {                                                              \
    F x = ld<F>(a), y = ld<F>(b), r;                             \
    switch (op) {                                                \
      case 0: r = fp_add(x, y); break;                           \
      case 1: r = fp_sub(x, y); break;                           \
      case 2: r = fp_mul(x, y); break;                           \
      case 3: r = fp_neg(x); break;                              \
      case 4: r = fp_inv(x); break;                              \
      case 5: r = fp_to_mont(x); break;                          \
      case 6: r = fp_from_mont(x); break;                        \
      case 7: r = fp_dbl(x); break;                              \
      case 8: r = fp_sqr(x); break;                              \
      case 9: r = fp_inv_gcd(x); break;                          \
      case 10: r = fp_inv_plain_gcd(x); break;                   \
      default: return -1;                                        \
    }                                                            \
    st(out, r);                                                  \
  }
  if (field == 0) RUN(Fr) else RUN(Fq)
  return 0;
}

// The wide-product building blocks of field.cuh.  a, b, c, d: 8 limbs each; t: 16 limbs; out: 16 limbs (ops 0, 1, 4)
// or 8 (ops 2, 3).  op: 0 out = a b, 1 out = a^2, 2 out = redc(t), 3 out = (a b + c d) R^-1, 4 out = t + a b with the
// carry limb as the return value ; field: 0 Fr, 1 Fq.  Returns -1 on a bad op.
int hs_wide_op(int field, int op, const uint32_t* a, const uint32_t* b, const uint32_t* c, const uint32_t* d,
               const uint32_t* t, uint32_t* out) {
#define RUN_WIDE(F, P)                                                        \
  {                                                                           \
    F x = ld<F>(a), y = ld<F>(b), z = ld<F>(c), u = ld<F>(d);                 \
    uint32_t T[16];                                                           \
    memcpy(T, t, sizeof(T));                                                  \
    switch (op) {                                                             \
      case 0: fp_mul_wide(T, x, y); break;                                    \
      case 1: fp_sqr_wide(T, x); break;                                       \
      case 2: st(out, fp_redc<P>(T)); return 0;                               \
      case 3: st(out, fp_mul_sum2(x, y, z, u)); return 0;                     \
      case 4: {                                                               \
        const uint32_t carry = fp_mad_wide(T, x, y);                          \
        memcpy(out, T, sizeof(T));                                            \
        return (int)carry;                                                    \
      }                                                                       \
      default: return -1;                                                     \
    }                                                                         \
    memcpy(out, T, sizeof(T));                                                \
  }
  if (field == 0) RUN_WIDE(Fr, FrParams) else RUN_WIDE(Fq, FqParams)
#undef RUN_WIDE
  return 0;
}

// The join of the slab-sharded NTT (ntt_shard.cuh): out[k] = sum_r x[r] w^(r k) for G = 2^log_g elements in Montgomery
// form, tw = w^0 .. w^(G/2 - 1) (Montgomery).  x, out: G x 8 limbs; tw: 4 x 8 limbs.
int hs_small_dft(int log_g, const uint32_t* x, const uint32_t* tw, uint32_t* out) {
  DftTw t;
  for (int k = 0; k < 4; k++) t.w[k] = ld<Fr>(tw + 8 * k);
#define RUN_DFT(LG)                                                     \
  {                                                                     \
    Fr v[1 << LG];                                                      \
    for (int i = 0; i < (1 << LG); i++) v[i] = ld<Fr>(x + 8 * i);       \
    small_dft<LG>(v, t);                                                \
    for (int i = 0; i < (1 << LG); i++) st(out + 8 * i, v[i]);          \
  }
  switch (log_g) {
    case 1: RUN_DFT(1) break;
    case 2: RUN_DFT(2) break;
    case 3: RUN_DFT(3) break;
    default: return -1;
  }
#undef RUN_DFT
  return 0;
}

// signed digits of a canonical scalar for window size c: writes W = ceil(256 / c) digits (sign * magnitude) and
// returns the carry left after the last window (must be 0 for scalars < r)
int hs_msm_digits(const uint32_t* scalar, uint32_t c, int32_t* digits, uint32_t* n_windows) {
  MsmGeom g;
  g.c = c;
  g.W = (256 + c - 1) / c;
  g.half = 1u << (c - 1);
  g.fixed_base = 0;
  g.point_stride = 0;
  g.batch = 1;
  g.lo = 0;
  g.nloc = g.half;
  g.own_log = 0;
  g.own_rank = 0;
  g.sets = g.W;
  g.nb = g.half * g.W;
  Fr s = ld<Fr>(scalar);
  DigitWalk dw(&s, 0, 0);
  for (uint32_t w = 0; w < g.W; w++) {
    uint32_t neg, d = dw.next(w, g, neg);
    digits[w] = neg ? -(int32_t)d : (int32_t)d;
  }
  *n_windows = g.W;
  return (int)dw.carry;
}

// G1 ops on Montgomery-form coordinates.  xyzz: 4x8 limbs (X, Y, ZZ, ZZZ); affine: 2x8 limbs + inf flag.
// op: 0 xyzz += affine, 1 xyzz += xyzz, 2 double, 3 to_affine
int hs_curve_op(int op, const uint32_t* acc_in, const uint32_t* other, int other_inf, uint32_t* out) {
  G1XYZZ acc;
  memcpy(&acc, acc_in, sizeof(acc));
  switch (op) {
    case 0: {
      G1Affine p;
      memcpy(&p.x, other, 32);
      memcpy(&p.y, other + 8, 32);
      if (!other_inf) g1_add_mixed(acc, p);
      break;
    }
    case 4: {
      G1Affine p;
      memcpy(&p.x, other, 32);
      memcpy(&p.y, other + 8, 32);
      if (!other_inf) g1_add_mixed_uniform(acc, p);
      break;
    }
    case 1: {
      G1XYZZ q;
      memcpy(&q, other, sizeof(q));
      g1_add(acc, q);
      break;
    }
    case 2: g1_double(acc); break;
    case 5: {
      G1XYZZ q;
      memcpy(&q, other, sizeof(q));
      g1_add_uniform(acc, q);
      break;
    }
    case 3: {
      G1Affine p;
      bool inf = g1_to_affine(acc, p);
      memcpy(out, &p.x, 32);
      memcpy(out + 8, &p.y, 32);
      return inf ? 1 : 0;
    }
    default: return -1;
  }
  memcpy(out, &acc, sizeof(acc));
  return 0;
}

// The whole bucket pipeline of msm.cu on the CPU, every thread body run in a loop: signed-digit slicing, histogram,
// padded scan, counting-sort scatter, rounds of batched affine additions (msm_bucket.cuh), recursive bucket reduction,
// bucket-range offset and window Horner.  points: n canonical affine points (16 words each); scalars: batch * n
// canonical scalars; fixed_base != 0 builds the window table 2^(c w) P_i first (batch <= 4 scalar vectors share it).
// [lo, hi): the bucket magnitudes this "rank" owns.  out: one canonical affine point (+ identity flag) per scalar
// vector: the rank's partial sum.  Returns the number of accumulation rounds that did work, -1 on bad input.
int hs_msm_pipeline(const uint32_t* points, uint32_t n, const uint32_t* scalars, uint32_t batch, uint32_t c,
                    int fixed_base, uint32_t lo, uint32_t hi, uint32_t B, uint32_t g0, uint32_t* out, uint8_t* out_inf) {
  if (!n || !batch || batch > 4 || (!fixed_base && batch != 1) || c < 1 || c > 16 || B < 2 || B > PB_AFF_BMAX) return -1;
  if (g0 < 2 || (g0 & (g0 - 1))) return -1;
  MsmGeom g;
  g.c = c;
  g.W = (256 + c - 1) / c;
  g.half = 1u << (c - 1);
  g.fixed_base = fixed_base ? 1 : 0;
  g.point_stride = fixed_base ? n : 0;
  g.batch = batch;
  g.own_log = 0;
  g.own_rank = 0;
  if (hi >= 0xfffffff0u && hi != 0xffffffffu) {  // strided shard: 2^(0xffffffff - hi) ranks, rank = lo
    g.own_log = 0xffffffffu - hi;
    g.own_rank = lo;
    g.lo = 0;
    g.nloc = g.half >> g.own_log;
    if (!g.nloc || lo >= (1u << g.own_log)) return -1;
  } else {
    if (hi > g.half) hi = g.half;
    if (lo >= hi) return -1;
    g.lo = lo;
    g.nloc = hi - lo;
  }
  g.sets = fixed_base ? batch : g.W;
  g.nb = g.sets * g.nloc;
  // point table
  std::vector<G1Affine> tab(fixed_base ? (size_t)g.W * n : n);
  for (uint32_t i = 0; i < n; i++) {
    tab[i].x = fp_to_mont(ld<Fq>(points + 16 * i));
    tab[i].y = fp_to_mont(ld<Fq>(points + 16 * i + 8));
  }
  if (fixed_base)
    for (uint32_t w = 1; w < g.W; w++)
      for (uint32_t i = 0; i < n; i++) {
        G1XYZZ a;
        g1_double_affine(a, tab[(size_t)(w - 1) * n + i]);
        for (uint32_t k = 1; k < c; k++) g1_double(a);
        g1_to_affine(a, tab[(size_t)w * n + i]);
      }
  std::vector<Fr> sc((size_t)batch * n);
  for (size_t i = 0; i < sc.size(); i++) sc[i] = ld<Fr>(scalars + 8 * i);
  // histogram, padded scan, scatter
  std::vector<uint32_t> counts(g.nb + 1, 0), off(g.nb + 1, 0), cursors(g.nb, 0);
  for (uint32_t k = 0; k < batch; k++)
    for (uint32_t i = 0; i < n; i++) {
      DigitWalk dw(sc.data() + (size_t)k * n, i, 0);
      for (uint32_t w = 0; w < g.W; w++) {
        uint32_t neg, d = dw.next(w, g, neg);
        if (!d) continue;
        uint32_t key = msm_bucket_key(g, k, w, d);
        if (key != 0xffffffffu) counts[key]++;
      }
    }
  uint32_t maxc = 0;
  for (uint32_t b = 0; b < g.nb; b++) { off[b + 1] = off[b] + ((counts[b] + 1) & ~1u); maxc = std::max(maxc, counts[b]); }
  counts[g.nb] = maxc;
  std::vector<uint32_t> sorted(off[g.nb] + 2, PB_MSM_PAD);
  for (uint32_t k = 0; k < batch; k++)
    for (uint32_t i = 0; i < n; i++) {
      DigitWalk dw(sc.data() + (size_t)k * n, i, 0);
      for (uint32_t w = 0; w < g.W; w++) {
        uint32_t neg, d = dw.next(w, g, neg);
        if (!d) continue;
        uint32_t key = msm_bucket_key(g, k, w, d);
        if (key == 0xffffffffu) continue;
        sorted[off[key] + cursors[key]++] = (uint32_t)((uint64_t)w * g.point_stride + i) | (neg << 31);
      }
    }
  // accumulation rounds
  const uint64_t positions = (uint64_t)n * g.W * batch + g.nb, s_bound = positions / 2;
  std::vector<G1Affine> pts(s_bound + 1);
  AffAcc a;
  a.table = tab.data();
  a.sorted = sorted.data();
  a.pts = pts.data();
  a.off = off.data();
  a.cnt = counts.data();
  a.max_cnt = counts.data() + g.nb;
  a.nbl = g.nb;
  a.B = B;
  Fq pref[PB_AFF_BMAX];
  uint32_t desc[PB_AFF_BMAX];
  int rounds = 0;
  for (uint32_t r = 0; r < 32; r++) {
    a.r = r;
    if (r > 0 && maxc > (1u << r)) rounds = r + 1;
    if (r == 0) rounds = 1;
    const uint64_t T = aff_round_threads(s_bound, B, r) + 40;  // spare threads must do nothing
    // descending thread order: a right-hand slot read late must still be intact (it is never written in its round)
    for (uint64_t t = T; t-- > 0;) {
      if (r == 0) aff_round0_thread(a, t, pref, desc);
      else aff_round_thread(a, t, pref, desc);
    }
  }
  // reduction
  ReduceArgs ra;
  ra.pts = pts.data(); ra.off = off.data(); ra.cnt = counts.data(); ra.xb = nullptr;
  ra.sets = g.sets; ra.m = g.nloc; ra.g = g0;
  std::vector<SR> cur((size_t)g.sets * reduce_groups(ra.m, ra.g)), nxt;
  ra.out = cur.data();
  for (uint64_t t = 0; t < cur.size() + 3; t++) reduce_level0_thread(ra, t);
  uint32_t m = reduce_groups(ra.m, ra.g), log_G = 0;
  while ((1u << log_G) < g0) log_G++;
  while (m > 8) {
    // the block-wide level (k_reduce_block in msm.cu), its phases run thread by thread
    const uint32_t chunks = reduce_chunks(m);
    nxt.assign((size_t)g.sets * chunks, SR());
    BlockLevelArgs ba;
    ba.in = cur.data(); ba.out = nxt.data(); ba.sets = g.sets; ba.m = m; ba.log_G = log_G;
    for (uint32_t set = 0; set < g.sets; set++)
      for (uint32_t chunk = 0; chunk < chunks; chunk++) {
        const uint32_t NT = PB_REDUCE_THREADS;
        std::vector<G1XYZZ> sh(NT), xs(NT), tmp(NT);
        for (uint32_t t = 0; t < NT; t++) blk_local(ba, set, chunk, t, sh[t], xs[t]);
        for (uint32_t d = 1; d < NT; d <<= 1) {
          for (uint32_t t = 0; t < NT; t++) tmp[t] = blk_scan_step(sh.data(), t, d);
          sh = tmp;
        }
        const G1XYZZ s_total = sh[0];
        for (uint32_t t = 0; t < NT; t++) tmp[t] = blk_weight(ba, t, xs[t], sh[t]);
        sh = tmp;
        for (uint32_t d = NT / 2; d > 0; d >>= 1)
          for (uint32_t t = 0; t < NT; t++) blk_tree_step(sh.data(), t, d);
        nxt[(size_t)set * chunks + chunk].S = s_total;
        nxt[(size_t)set * chunks + chunk].R = sh[0];
      }
    m = chunks;
    log_G += 9;
    cur.swap(nxt);
  }
  {  // the last <= 8 elements of every set: folded by the host code of msm.cu
    std::vector<SR> fin(g.sets);
    for (uint32_t s = 0; s < g.sets; s++) fin[s] = reduce_fold_final(cur.data() + (size_t)s * m, m, log_G);
    cur.swap(fin);
  }
  std::vector<G1XYZZ> ws(g.sets);
  for (uint32_t s = 0; s < g.sets; s++) {
    if (g.own_log) {  // strided shard: sum_k (G k + r + 1) B_k = G R + (r + 1 - G) S
      std::vector<SR> one(1, cur[s]);
      // a one-rank "join" with the rank's own coefficient: reuse the library's formula through its pieces
      G1XYZZ gr = cur[s].R;
      for (uint32_t k = 0; k < g.own_log; k++) g1_double(gr);
      G1XYZZ ms = G1XYZZ::identity();
      const uint32_t coef = (1u << g.own_log) - 1 - g.own_rank;  // subtract (G - 1 - r) S
      for (int i = 31; i >= 0; i--) { g1_double(ms); if ((coef >> i) & 1) g1_add(ms, cur[s].S); }
      ms.Y = fp_neg(ms.Y);
      g1_add(gr, ms);
      ws[s] = gr;
      continue;
    }
    ws[s] = cur[s].R;
    G1XYZZ ml = G1XYZZ::identity();
    for (int i = 31; i >= 0; i--) { g1_double(ml); if ((g.lo >> i) & 1) g1_add(ml, cur[s].S); }
    g1_add(ws[s], ml);
  }
  auto emit = [&](const G1XYZZ& r, uint32_t k) {
    G1Affine p;
    bool inf = g1_to_affine(r, p);
    out_inf[k] = inf ? 1 : 0;
    Fq x = fp_from_mont(p.x), y = fp_from_mont(p.y);
    st(out + 16 * k, x);
    st(out + 16 * k + 8, y);
  };
  if (fixed_base) {
    for (uint32_t k = 0; k < batch; k++) emit(ws[k], k);
  } else {
    G1XYZZ r = G1XYZZ::identity();
    for (int w = (int)g.W - 1; w >= 0; w--) {
      if (w != (int)g.W - 1) for (uint32_t k = 0; k < c; k++) g1_double(r);
      g1_add(r, ws[w]);
    }
    emit(r, 0);
  }
  return rounds;
}
}
