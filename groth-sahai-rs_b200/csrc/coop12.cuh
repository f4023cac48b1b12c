// Cooperative Fp12 arithmetic: ONE WARP PER w-POWER COEFFICIENT, ONE LANE PER ACCUMULATOR.
//
// A block of 6 warps (192 threads) owns 32 independent Fp12 values  f = sum_{k<6} a_k w^k  (a_k in Fp2,
// w^6 = xi = 1 + u; a_0=c0.c0, a_1=c1.c0, a_2=c0.c1, a_3=c1.c1, a_4=c0.c2, a_5=c1.c2 of the tower form).
// Warp k computes output coefficient k of all 32 values, so every k-dependent decision (which inputs,
// where xi is applied) is warp-uniform and all 32 lanes stay busy.  The values live in SHARED memory in
// the "Q layout" (below); each output coefficient is produced as a SUM OF Fp2 PRODUCTS with lazy reduction:
//     r.c0 = sum_t ( Y_t.c0 * X_t.c0 - Y_t.c1 * X_t.c1 )        one interleaved Montgomery reduction
//     r.c1 = sum_t ( Y_t.c0 * X_t.c1 + Y_t.c1 * X_t.c0 )        per Fp component (fp.cuh rowsum_l)
// with the Y operands held in registers (2 x 12 limbs per term) and the X operands streamed limb-quad by
// limb-quad out of shared memory (LDS.128, conflict free).  No temporaries outside registers, no local memory.
//
// Every op reads one accumulator buffer and writes another one (ping-pong), so a single block barrier per op
// is enough.  The functions are plain (k, lane) functions over word arrays so that tests/hostsim can run the
// identical code on the CPU by looping over (k, lane) between "barriers".
//
// Replaces: ark-ff Fp12 multiplication / squaring / sparse line multiplication underneath
// E::multi_miller_loop and E::final_exponentiation (reference call sites src/data_structures.rs:484-502).
#pragma once
#include "tower.cuh"

namespace gs {

constexpr int CQ_LANES = 32;
constexpr int CQ_QUAD = 4 * CQ_LANES;  // words per limb-quad of one Fp over the 32 lanes
constexpr int CQ_FP = 12 * CQ_LANES;   // words per Fp over the 32 lanes: [quad 0..2][lane][4]
constexpr int CQ_ACC = 12 * CQ_FP;     // one Fp12 accumulator set: Fp index = 2*coef + component

struct alignas(16) q4 {
  uint32_t v[4];
};

// pointer to quad 0 of Fp number `idx` of lane `lane`
GS_HD GS_INL const uint32_t* cq_ptr(const uint32_t* base, int idx, int lane) { return base + idx * CQ_FP + lane * 4; }
GS_HD GS_INL uint32_t* cq_ptr(uint32_t* base, int idx, int lane) { return base + idx * CQ_FP + lane * 4; }

GS_HD GS_INL void cq_ld(fp& r, const uint32_t* p) {
#pragma unroll
  for (int q = 0; q < 3; q++) {
    q4 t = *(const q4*)(p + q * CQ_QUAD);
#pragma unroll
    for (int i = 0; i < 4; i++) r.l[q * 4 + i] = t.v[i];
  }
}
GS_HD GS_INL void cq_st(uint32_t* p, const fp& a) {
#pragma unroll
  for (int q = 0; q < 3; q++) {
    q4 t;
#pragma unroll
    for (int i = 0; i < 4; i++) t.v[i] = a.l[q * 4 + i];
    *(q4*)(p + q * CQ_QUAD) = t;
  }
}

// r = (sum_t a[t] * B_t) / R mod p, B_t streamed from the Q layout (b[t] = pointer to quad 0 of this lane)
template <int NT>
GS_HD GS_INL void mulsum_q(fp& r, const fp (&a)[NT], const uint32_t* const (&b)[NT]) {
  uint32_t E[12], O[12];
#pragma unroll
  for (int q = 0; q < 3; q++) {
    q4 bl[NT];
#pragma unroll
    for (int t = 0; t < NT; t++) bl[t] = *(const q4*)(b[t] + q * CQ_QUAD);
#pragma unroll
    for (int ii = 0; ii < 4; ii++) {
      uint32_t lim[NT];
#pragma unroll
      for (int t = 0; t < NT; t++) lim[t] = bl[t].v[ii];
      if ((ii & 1) == 0)
        fp::rowsum_l<NT>(E, O, a, lim, q == 0 && ii == 0);
      else
        fp::rowsum_l<NT>(O, E, a, lim, false);
    }
  }
  fp::mulsum_finish(r, E, O);
}

// r = sum_{t<NT} Y_t * X_t in Fp2.  y[2t], y[2t+1] = Y_t.c0, Y_t.c1 in registers (y[2t+1] is NEGATED on
// return); x0[t], x1[t] = Q-layout pointers of X_t.c0, X_t.c1.  All operands canonical; 2*NT <= 8.
template <int NT>
GS_HD GS_INL void cq_fp2_dot(fp2& r, fp (&y)[2 * NT], const uint32_t* const (&x0)[NT], const uint32_t* const (&x1)[NT]) {
  const uint32_t* b[2 * NT];
#pragma unroll
  for (int t = 0; t < NT; t++) {
    b[2 * t] = x1[t];
    b[2 * t + 1] = x0[t];
  }
  mulsum_q<2 * NT>(r.c1, y, b);
#pragma unroll
  for (int t = 0; t < NT; t++) {
    fp::neg(y[2 * t + 1], y[2 * t + 1]);
    b[2 * t] = x0[t];
    b[2 * t + 1] = x1[t];
  }
  mulsum_q<2 * NT>(r.c0, y, b);
}

// r = Y_0 X_0 + Y_1 X_1 in Fp2 by Karatsuba over BOTH products at once: three lazily reduced sums of two Fp products
//     P0 = sum Y_t.c0 X_t.c0,  P1 = sum Y_t.c1 X_t.c1,  P2 = sum (Y_t.c0 + Y_t.c1)(X_t.c0 + X_t.c1);  r = (P0 - P1, P2 - P0 - P1)
// 6 Fp products + 3 reductions (1,332 multiply-adds) instead of the 8 + 2 (1,464) of cq_fp2_dot<2>.  y[2t], y[2t+1] =
// Y_t.c0, Y_t.c1 in registers (unchanged); the X operands are read from the Q layout, their component sums formed in
// registers.
GS_HD GS_INL void cq_fp2_dot2_k(fp2& r, const fp (&y)[4], const uint32_t* const (&x0)[2], const uint32_t* const (&x1)[2]) {
  fp P0, P1, P2;
  {
    const fp a[2] = {y[0], y[2]};
    mulsum_q<2>(P0, a, x0);
  }
  {
    const fp a[2] = {y[1], y[3]};
    mulsum_q<2>(P1, a, x1);
  }
  {
    fp a[2], b[2], t0, t1;
    fp::add(a[0], y[0], y[1]);
    fp::add(a[1], y[2], y[3]);
    cq_ld(t0, x0[0]);
    cq_ld(t1, x1[0]);
    fp::add(b[0], t0, t1);
    cq_ld(t0, x0[1]);
    cq_ld(t1, x1[1]);
    fp::add(b[1], t0, t1);
    fp::mulsum<2>(P2, a, b);
  }
  fp::sub(r.c0, P0, P1);
  fp::sub(r.c1, P2, P0);
  fp::sub(r.c1, r.c1, P1);
}

// the same over three products (the two passes of cq_mul): 9 Fp products + 3 reductions (1,764 multiply-adds) instead of
// 12 + 2 (2,040).  The component sums of Y are formed first, so that Y itself is dead by the time P2 is computed.
GS_HD GS_INL void cq_fp2_dot3_k(fp2& r, const fp (&y)[6], const uint32_t* const (&x0)[3], const uint32_t* const (&x1)[3]) {
  fp P0, P1, P2, sa[3];
#pragma unroll
  for (int t = 0; t < 3; t++) fp::add(sa[t], y[2 * t], y[2 * t + 1]);
  {
    const fp a[3] = {y[0], y[2], y[4]};
    mulsum_q<3>(P0, a, x0);
  }
  {
    const fp a[3] = {y[1], y[3], y[5]};
    mulsum_q<3>(P1, a, x1);
  }
  {
    fp b[3];
#pragma unroll
    for (int t = 0; t < 3; t++) {
      fp t0, t1;
      cq_ld(t0, x0[t]);
      cq_ld(t1, x1[t]);
      fp::add(b[t], t0, t1);
    }
    fp::mulsum<3>(P2, sa, b);
  }
  fp::sub(r.c0, P0, P1);
  fp::sub(r.c1, P2, P0);
  fp::sub(r.c1, r.c1, P1);
}

// lo + hi R = sum_t a[t] * B_t unreduced (fp.cuh rowsum_w), B_t streamed from the Q layout: B_t = b0[t], or with SUM the
// limb-wise sum b0[t] + b1[t] (the carry of each quad is kept for the next one; both canonical, so B_t < 2p fits 12 limbs)
template <int NT, bool SUM>
GS_HD GS_INL void cq_mulsum_w(uint32_t (&lo)[12], uint32_t (&hi)[12], const fp (&a)[NT], const uint32_t* const (&b0)[NT],
                              const uint32_t* const (&b1)[NT]) {
  uint32_t E[12], O[12], cy[NT];
#pragma unroll
  for (int q = 0; q < 3; q++) {
    q4 bl[NT];
#pragma unroll
    for (int t = 0; t < NT; t++) {
      bl[t] = *(const q4*)(b0[t] + q * CQ_QUAD);
      if (SUM) {
        const q4 u = *(const q4*)(b1[t] + q * CQ_QUAD);
        if (q == 0)
          bl[t].v[0] = add_cc(bl[t].v[0], u.v[0]);
        else {
          add_cc(cy[t], 0xffffffffu);  // CC = carry out of the previous quad
          bl[t].v[0] = addc_cc(bl[t].v[0], u.v[0]);
        }
#pragma unroll
        for (int i = 1; i < 4; i++) bl[t].v[i] = addc_cc(bl[t].v[i], u.v[i]);
        cy[t] = addc(0u, 0u);
      }
    }
#pragma unroll
    for (int ii = 0; ii < 4; ii++) {
      uint32_t lim[NT];
#pragma unroll
      for (int t = 0; t < NT; t++) lim[t] = bl[t].v[ii];
      if ((ii & 1) == 0) {
        fp::rowsum_w<NT>(E, O, a, lim, q == 0 && ii == 0);
        lo[q * 4 + ii] = E[0];
      } else {
        fp::rowsum_w<NT>(O, E, a, lim, false);
        lo[q * 4 + ii] = O[0];
      }
    }
  }
  fp::window_out(hi, E, O);
}

// r = sum_{t<NT} Y_t X_t in Fp2 by Karatsuba with ONE Montgomery reduction per output component.  The three sums
//     P0 = sum Y_t.c0 X_t.c0,   P1 = sum Y_t.c1 X_t.c1,   P2 = sum (Y_t.c0 + Y_t.c1)(X_t.c0 + X_t.c1)
// are formed as unreduced 24-limb integers, with the component sums NOT reduced, so that exactly
//     P2 - P0 - P1 = sum (Y_t.c0 X_t.c1 + Y_t.c1 X_t.c0),  in [0, 2 NT p^2)
// and r.c1 = REDC(P2 - (P0 + P1)), r.c0 = REDC(P0 - P1 + K) with K = p 2^383 (4.92 p^2 > NT p^2 > P1, a multiple of p, so
// the argument is >= 0 and congruent to P0 - P1).  Both arguments stay below 2 NT p^2 + 4.92 p^2 < p R = 9.84 p^2 for
// NT <= 4, the bound of fp::redc_w, whose canonical result is therefore the one every other form produces.  The
// rowsum_w windows need sum_t a[t] < R: at most 2 NT p < R for the component sums.
// 3 NT Fp products + 2 reductions (NT = 2: 1,176 multiply-adds against the 1,332 of three reduced sums).
// ld(a, c) fills a[t] with Y_t.c0 (c = 0), Y_t.c1 (c = 1), each canonical, or (c = 2) their plain integer sum
// Y_t.c0 + Y_t.c1 of exactly those values; X_t.c0, X_t.c1 (canonical) are read from the Q layout.
template <int NT, class LD>
GS_HD GS_INL void cq_fp2_dot_w(fp2& r, LD ld, const uint32_t* const (&x0)[NT], const uint32_t* const (&x1)[NT]) {
  static_assert(NT >= 1 && NT <= 4, "bounds above hold for NT <= 4");
  uint32_t slo[12], shi[12];
  {
    uint32_t lo0[12], hi0[12], lo1[12], hi1[12];
    {
      fp a[NT];
      ld(a, 0);
      cq_mulsum_w<NT, false>(lo0, hi0, a, x0, x0);
    }
    {
      fp a[NT];
      ld(a, 1);
      cq_mulsum_w<NT, false>(lo1, hi1, a, x1, x1);
    }
    // S = P0 + P1 (< 2 NT p^2 < 2^768),  D = P0 - P1 + K (the subtraction may wrap mod 2^768; adding K unwraps it)
    uint32_t dlo[12], dhi[12];
    slo[0] = add_cc(lo0[0], lo1[0]);
#pragma unroll
    for (int i = 1; i < 12; i++) slo[i] = addc_cc(lo0[i], lo1[i]);
#pragma unroll
    for (int i = 0; i < 11; i++) shi[i] = addc_cc(hi0[i], hi1[i]);
    shi[11] = addc(hi0[11], hi1[11]);
    dlo[0] = sub_cc(lo0[0], lo1[0]);
#pragma unroll
    for (int i = 1; i < 12; i++) dlo[i] = subc_cc(lo0[i], lo1[i]);
#pragma unroll
    for (int i = 0; i < 11; i++) dhi[i] = subc_cc(hi0[i], hi1[i]);
    dhi[11] = subc(hi0[11], hi1[11]);
    // K = p << 383: limbs 11..23 = (p[j] << 31) | (p[j-1] >> 1)
    dlo[11] = add_cc(dlo[11], FpParams::mod(0) << 31);
#pragma unroll
    for (int j = 1; j < 12; j++) dhi[j - 1] = addc_cc(dhi[j - 1], (FpParams::mod(j) << 31) | (FpParams::mod(j - 1) >> 1));
    dhi[11] = addc(dhi[11], FpParams::mod(11) >> 1);
    fp::redc_w(r.c0, dlo, dhi);
  }
  {
    uint32_t lo2[12], hi2[12];
    {
      fp a[NT];
      ld(a, 2);
      cq_mulsum_w<NT, true>(lo2, hi2, a, x0, x1);
    }
    lo2[0] = sub_cc(lo2[0], slo[0]);
#pragma unroll
    for (int i = 1; i < 12; i++) lo2[i] = subc_cc(lo2[i], slo[i]);
#pragma unroll
    for (int i = 0; i < 11; i++) hi2[i] = subc_cc(hi2[i], shi[i]);
    hi2[11] = subc(hi2[11], shi[11]);
    fp::redc_w(r.c1, lo2, hi2);
  }
}

// register-side operands of cq_fp2_dot_w held in registers: y[2t], y[2t+1] = Y_t.c0, Y_t.c1
template <int NT>
struct cq_yreg {
  const fp (&y)[2 * NT];
  GS_HD GS_INL void operator()(fp (&a)[NT], int c) const {
#pragma unroll
    for (int t = 0; t < NT; t++) {
      if (c < 2)
        a[t] = y[2 * t + c];
      else
        fp::add_noreduce(a[t], y[2 * t], y[2 * t + 1]);
    }
  }
};

// load coefficient j of the accumulator set `f` into (y0, y1), optionally times xi and/or 2
GS_HD GS_INL void cq_ld_coef(fp& y0, fp& y1, const uint32_t* f, int j, int lane, bool xi, bool dbl) {
  cq_ld(y0, cq_ptr(f, 2 * j, lane));
  cq_ld(y1, cq_ptr(f, 2 * j + 1, lane));
  if (xi) {
    fp t0, t1;
    fp::sub(t0, y0, y1);
    fp::add(t1, y0, y1);
    y0 = t0;
    y1 = t1;
  }
  if (dbl) {
    fp::add(y0, y0, y0);
    fp::add(y1, y1, y1);
  }
}
GS_HD GS_INL void cq_st_coef(uint32_t* f, int k, int lane, const fp2& r) {
  cq_st(cq_ptr(f, 2 * k, lane), r.c0);
  cq_st(cq_ptr(f, 2 * k + 1, lane), r.c1);
}

// ------------------------------------------------------------------ sparse line multiplication
// fout.a_k = alpha a_k + beta a_{k-2} + gamma a_{k-3}   (indices mod 6, times xi on wrap-around), i.e.
// f * (alpha + beta w^2 + gamma w^3): the M-twist line  (= ark-ff mul_by_014 in the w basis).
// `tile` holds alpha.c0, alpha.c1, beta.c0, beta.c1, gamma.c0, gamma.c1 (6 Fp, Q layout).
// !active lanes copy their coefficient through unchanged (pair dropped: identity on either side).
GS_HD GS_INL void cq_line_mul(int k, int lane, const uint32_t* fin, uint32_t* fout, const uint32_t* tile, bool active) {
  fp y[6];
  const int j1 = k >= 2 ? k - 2 : k + 4, j2 = k >= 3 ? k - 3 : k + 3;
  cq_ld_coef(y[0], y[1], fin, k, lane, false, false);
  cq_ld_coef(y[2], y[3], fin, j1, lane, k < 2, false);
  cq_ld_coef(y[4], y[5], fin, j2, lane, k < 3, false);
  const uint32_t* x0[3] = {cq_ptr(tile, 0, lane), cq_ptr(tile, 2, lane), cq_ptr(tile, 4, lane)};
  const uint32_t* x1[3] = {cq_ptr(tile, 1, lane), cq_ptr(tile, 3, lane), cq_ptr(tile, 5, lane)};
  fp2 r;
  cq_fp2_dot<3>(r, y, x0, x1);
  if (!active) cq_ld_coef(r.c0, r.c1, fin, k, lane, false, false);
  cq_st_coef(fout, k, lane, r);
}

// Same with gamma = 1 (affine line scaled by 1/yP, pairing.cuh g2_affine_step):
//     fout.a_k = alpha a_k + beta a_{k-2} + a_{k-3}
// `tile` holds alpha.c0, alpha.c1, beta.c0, beta.c1 (4 Fp): a two-term Fp2 dot product per coefficient instead of three,
// and only two register-side operands.
// GS_LINE_KARATSUBA selects the form of the dot products here and in cq_sqr: 0 = schoolbook (cq_fp2_dot), 1 = Karatsuba
// with three reduced sums (cq_fp2_dot2_k), 2 = Karatsuba with one reduction per component (cq_fp2_dot_w).
#ifndef GS_LINE_KARATSUBA
#define GS_LINE_KARATSUBA 2
#endif
GS_HD GS_INL void cq_line_mul_u(int k, int lane, const uint32_t* fin, uint32_t* fout, const uint32_t* tile, bool active) {
  fp y[4];
  const int j1 = k >= 2 ? k - 2 : k + 4, j2 = k >= 3 ? k - 3 : k + 3;
  cq_ld_coef(y[0], y[1], fin, k, lane, false, false);
  cq_ld_coef(y[2], y[3], fin, j1, lane, k < 2, false);
  fp2 r, u;
  const uint32_t* x0[2] = {cq_ptr(tile, 0, lane), cq_ptr(tile, 2, lane)};
  const uint32_t* x1[2] = {cq_ptr(tile, 1, lane), cq_ptr(tile, 3, lane)};
#if GS_LINE_KARATSUBA == 2
  cq_fp2_dot_w<2>(r, cq_yreg<2>{y}, x0, x1);
#elif GS_LINE_KARATSUBA == 1
  cq_fp2_dot2_k(r, y, x0, x1);
#else
  cq_fp2_dot<2>(r, y, x0, x1);
#endif
  cq_ld_coef(u.c0, u.c1, fin, j2, lane, k < 3, false);
  fp2::add(r, r, u);
  if (!active) cq_ld_coef(r.c0, r.c1, fin, k, lane, false, false);
  cq_st_coef(fout, k, lane, r);
}

// ------------------------------------------------------------------ squaring
// fout = fin^2:  b_k = sum_{i<=j, i+j = k mod 6} c_ij a_i a_j,  c_ij = (i<j ? 2 : 1) * (i+j >= 6 ? xi : 1).
// Even k have 4 terms (2 doubled pairs + 2 squares), odd k have 3 doubled pairs; two passes of <= 2 terms (one pass over
// all four terms needs more than the 168 registers k_miller4 has).
GS_HD GS_INL void cq_sqr(int k, int lane, const uint32_t* fin, uint32_t* fout) {
  int ti[4], tj[4], nt = 0;
  for (int i = 0; i < 6; i++) {
    int j = (k - i + 6) % 6;
    if (i <= j) {
      ti[nt] = i;
      tj[nt] = j;
      nt++;
    }
  }
  fp2 r, r2;
  {
    fp y[4];
    cq_ld_coef(y[0], y[1], fin, tj[0], lane, ti[0] + tj[0] >= 6, ti[0] < tj[0]);
    cq_ld_coef(y[2], y[3], fin, tj[1], lane, ti[1] + tj[1] >= 6, ti[1] < tj[1]);
    const uint32_t* x0[2] = {cq_ptr(fin, 2 * ti[0], lane), cq_ptr(fin, 2 * ti[1], lane)};
    const uint32_t* x1[2] = {cq_ptr(fin, 2 * ti[0] + 1, lane), cq_ptr(fin, 2 * ti[1] + 1, lane)};
#if GS_LINE_KARATSUBA == 2
    cq_fp2_dot_w<2>(r, cq_yreg<2>{y}, x0, x1);
#elif GS_LINE_KARATSUBA == 1
    cq_fp2_dot2_k(r, y, x0, x1);
#else
    cq_fp2_dot<2>(r, y, x0, x1);
#endif
    cq_st_coef(fout, k, lane, r);  // parked in the output slot (nobody reads fout during this op)
  }
  if (nt == 4) {
    fp y[4];
    cq_ld_coef(y[0], y[1], fin, tj[2], lane, ti[2] + tj[2] >= 6, ti[2] < tj[2]);
    cq_ld_coef(y[2], y[3], fin, tj[3], lane, ti[3] + tj[3] >= 6, ti[3] < tj[3]);
    const uint32_t* x0[2] = {cq_ptr(fin, 2 * ti[2], lane), cq_ptr(fin, 2 * ti[3], lane)};
    const uint32_t* x1[2] = {cq_ptr(fin, 2 * ti[2] + 1, lane), cq_ptr(fin, 2 * ti[3] + 1, lane)};
#if GS_LINE_KARATSUBA == 2
    cq_fp2_dot_w<2>(r2, cq_yreg<2>{y}, x0, x1);
#elif GS_LINE_KARATSUBA == 1
    cq_fp2_dot2_k(r2, y, x0, x1);
#else
    cq_fp2_dot<2>(r2, y, x0, x1);
#endif
  } else {
    fp y[2];
    cq_ld_coef(y[0], y[1], fin, tj[2], lane, ti[2] + tj[2] >= 6, ti[2] < tj[2]);
    const uint32_t* x0[1] = {cq_ptr(fin, 2 * ti[2], lane)};
    const uint32_t* x1[1] = {cq_ptr(fin, 2 * ti[2] + 1, lane)};
#if GS_LINE_KARATSUBA == 2
    cq_fp2_dot_w<1>(r2, cq_yreg<1>{y}, x0, x1);
#else
    cq_fp2_dot<1>(r2, y, x0, x1);
#endif
  }
  cq_ld_coef(r.c0, r.c1, fout, k, lane, false, false);
  fp2::add(r, r, r2);
  cq_st_coef(fout, k, lane, r);
}

// ------------------------------------------------------------------ general product
// fout = f * g:  b_k = sum_i g_i f_{k-i}  (xi on wrap-around).  f on the register side, g streamed.
GS_HD GS_INL void cq_mul(int k, int lane, const uint32_t* f, const uint32_t* g, uint32_t* fout) {
  fp2 r, r2;
#pragma unroll 1
  for (int h = 0; h < 2; h++) {
    fp y[6];
    const uint32_t *x0[3], *x1[3];
#pragma unroll
    for (int t = 0; t < 3; t++) {
      int i = h * 3 + t;
      int j = (k - i + 6) % 6;
      cq_ld_coef(y[2 * t], y[2 * t + 1], f, j, lane, i > k, false);
      x0[t] = cq_ptr(g, 2 * i, lane);
      x1[t] = cq_ptr(g, 2 * i + 1, lane);
    }
// GS_MUL_KARATSUBA: 0 = schoolbook, 1 = three reduced sums (cq_fp2_dot3_k), 2 = one reduction per component
#ifndef GS_MUL_KARATSUBA
#define GS_MUL_KARATSUBA 2
#endif
    if (h == 0) {
#if GS_MUL_KARATSUBA == 2
      cq_fp2_dot_w<3>(r, cq_yreg<3>{y}, x0, x1);
#elif GS_MUL_KARATSUBA == 1
      cq_fp2_dot3_k(r, y, x0, x1);
#else
      cq_fp2_dot<3>(r, y, x0, x1);
#endif
      cq_st_coef(fout, k, lane, r);  // parked in the output slot
    } else {
#if GS_MUL_KARATSUBA == 2
      cq_fp2_dot_w<3>(r2, cq_yreg<3>{y}, x0, x1);
#elif GS_MUL_KARATSUBA == 1
      cq_fp2_dot3_k(r2, y, x0, x1);
#else
      cq_fp2_dot<3>(r2, y, x0, x1);
#endif
    }
  }
  cq_ld_coef(r.c0, r.c1, fout, k, lane, false, false);
  fp2::add(r, r, r2);
  cq_st_coef(fout, k, lane, r);
}

// ------------------------------------------------------------------ cyclotomic squaring (Granger-Scott)
// For f in the cyclotomic subgroup, with the Fp4 pairs (x, y) = (a_0,a_3), (a_1,a_4), (a_2,a_5) (y on w^3):
//     S_g = x^2 + xi y^2,  P_g = 2 x y     and
//     a_0' = 3 S_0 - 2 a_0   a_3' = 3 P_0 + 2 a_3
//     a_2' = 3 S_1 - 2 a_2   a_5' = 3 P_1 + 2 a_5
//     a_4' = 3 S_2 - 2 a_4   a_1' = 3 xi P_2 + 2 a_1        (= ark-ff cyclotomic_square in the w basis)
// Balanced over the 6 warps by Fp COMPONENT: warp (g = k % 3, c = k / 3) computes component c of S_g and of P_g, each
// as ONE lazily reduced sum of products with BOTH operands in registers (the factors are sums / differences of the
// loaded coefficients, which the squaring structure allows):
//     S.c0 = (x0 + x1)(x0 - x1) + (y0 + y1)(y0 - y1) - (2 y0) y1        (xi y^2).c0 = y0^2 - y1^2 - 2 y0 y1
//     S.c1 = (2 x0) x1          + (y0 + y1)(y0 - y1) + (2 y0) y1        (xi y^2).c1 = y0^2 - y1^2 + 2 y0 y1
//     P.c0 = X0 y0 - X1 y1,  P.c1 = X0 y1 + X1 y0,  X = 2 x (times xi for g = 2)
// 3 + 2 Fp products and 2 reductions per warp (the schoolbook form with one operand streamed from shared memory took 4 + 2).
GS_HD GS_INL void cq_cyc_sqr(int k, int lane, const uint32_t* fin, uint32_t* fout) {
  const int g = k % 3, c = k / 3;
  const int ix = g, iy = g + 3;
  const int tS = g == 0 ? 0 : (g == 1 ? 2 : 4), tP = g == 0 ? 3 : (g == 1 ? 5 : 1);
  fp x0, x1, y0, y1;
  cq_ld_coef(x0, x1, fin, ix, lane, false, false);
  cq_ld_coef(y0, y1, fin, iy, lane, false, false);
  fp S, Pp;
  {
    fp a[3], b[3];
    fp::add(a[1], y0, y1);
    fp::sub(b[1], y0, y1);
    fp::add(a[2], y0, y0);
    b[2] = y1;
    if (c == 0) {
      fp::add(a[0], x0, x1);
      fp::sub(b[0], x0, x1);
      fp::neg(a[2], a[2]);
    } else {
      fp::add(a[0], x0, x0);
      b[0] = x1;
    }
    fp::mulsum<3>(S, a, b);
  }
  {
    fp a[2], b[2];
    if (g == 2) {
      fp::sub(a[0], x0, x1);
      fp::add(a[1], x0, x1);
    } else {
      a[0] = x0;
      a[1] = x1;
    }
    fp::add(a[0], a[0], a[0]);
    fp::add(a[1], a[1], a[1]);
    if (c == 0) {
      fp::neg(a[1], a[1]);
      b[0] = y0;
      b[1] = y1;
    } else {
      b[0] = y1;
      b[1] = y0;
    }
    fp::mulsum<2>(Pp, a, b);
  }
  fp t, o;
  // 3 S - 2 a_tS
  cq_ld(t, cq_ptr(fin, 2 * tS + c, lane));
  fp::sub(o, S, t);
  fp::add(o, o, o);
  fp::add(o, o, S);
  cq_st(cq_ptr(fout, 2 * tS + c, lane), o);
  // 3 P + 2 a_tP
  cq_ld(t, cq_ptr(fin, 2 * tP + c, lane));
  fp::add(o, Pp, t);
  fp::add(o, o, o);
  fp::add(o, o, Pp);
  cq_st(cq_ptr(fout, 2 * tP + c, lane), o);
}

// ------------------------------------------------------------------ coefficient-local ops (no cross-warp reads)
GS_HD GS_INL void cq_copy(int k, int lane, const uint32_t* fin, uint32_t* fout) {
  fp2 r;
  cq_ld_coef(r.c0, r.c1, fin, k, lane, false, false);
  cq_st_coef(fout, k, lane, r);
}
// conjugation x -> x^(p^6): negate the odd powers of w
GS_HD GS_INL void cq_conj(int k, int lane, const uint32_t* fin, uint32_t* fout) {
  fp2 r;
  cq_ld_coef(r.c0, r.c1, fin, k, lane, false, false);
  if (k & 1) fp2::neg(r, r);
  cq_st_coef(fout, k, lane, r);
}
// x -> x^(p^K), K = 1, 2:  (a_k w^k)^(p^K) = conj^K(a_k) * FROB_K[k] * w^k
template <int K>
GS_HD GS_INL void cq_frob(int k, int lane, const uint32_t* fin, uint32_t* fout) {
  fp2 t;
  cq_ld_coef(t.c0, t.c1, fin, k, lane, false, false);
  if (K & 1) fp::neg(t.c1, t.c1);
  if (k > 0) {
    fp2 g, r;
    for (int j = 0; j < 12; j++) {
      g.c0.l[j] = frob_coeff(K, k, 0, j);
      g.c1.l[j] = frob_coeff(K, k, 1, j);
    }
    fp s0, s1, t0, t1, t2;
    fp::add(s0, t.c0, t.c1);
    fp::add(s1, g.c0, g.c1);
    fp::mul(t0, t.c0, g.c0);
    fp::mul(t1, t.c1, g.c1);
    fp::mul(t2, s0, s1);
    fp::sub(r.c0, t0, t1);
    fp::sub(t2, t2, t0);
    fp::sub(r.c1, t2, t1);
    t = r;
  }
  cq_st_coef(fout, k, lane, t);
}
// fout = 1 / N for N in Fp6 = {a_0 + a_2 w^2 + a_4 w^4} (odd coefficients of fin ignored, of fout zeroed).
// Warp 0 inverts for its 32 lanes with the tower code (one Fermat inversion per lane); the others only zero.
GS_HD GS_INL void cq_inv6(int k, int lane, const uint32_t* fin, uint32_t* fout) {
  if (k == 0) {
    fp6 n, r;
    cq_ld_coef(n.c0.c0, n.c0.c1, fin, 0, lane, false, false);
    cq_ld_coef(n.c1.c0, n.c1.c1, fin, 2, lane, false, false);
    cq_ld_coef(n.c2.c0, n.c2.c1, fin, 4, lane, false, false);
    fp6::inv(r, n);
    cq_st_coef(fout, 0, lane, r.c0);
    cq_st_coef(fout, 2, lane, r.c1);
    cq_st_coef(fout, 4, lane, r.c2);
  } else if (k & 1) {
    fp2 z;
    z.set_zero();
    cq_st_coef(fout, k, lane, z);
  }
}

// ------------------------------------------------------------------ op programs
// A cooperative computation is a straight-line PROGRAM of ops over a small set of accumulator buffers; the
// kernel executes op after op with one block barrier in between, and tests/hostsim executes the same
// program by looping over (k, lane).  An op never reads a buffer it writes, except the coefficient-local
// ones (COPY / CONJ / FROB / INV6), which may run in place.
enum { CQ_OP_MUL = 1, CQ_OP_SQR, CQ_OP_CYC, CQ_OP_COPY, CQ_OP_CONJ, CQ_OP_FROB1, CQ_OP_FROB2, CQ_OP_INV6 };
GS_HD constexpr uint32_t cq_ins(int op, int dst, int a, int b = 0) {
  return (uint32_t)op | ((uint32_t)dst << 8) | ((uint32_t)a << 16) | ((uint32_t)b << 24);
}
GS_HD GS_INL void cq_exec(uint32_t ins, int k, int lane, uint32_t* bufs) {
  const int op = ins & 255;
  uint32_t* d = bufs + ((ins >> 8) & 255) * CQ_ACC;
  const uint32_t* a = bufs + ((ins >> 16) & 255) * CQ_ACC;
  const uint32_t* b = bufs + ((ins >> 24) & 255) * CQ_ACC;
  switch (op) {
    case CQ_OP_MUL: cq_mul(k, lane, a, b, d); break;
    case CQ_OP_SQR: cq_sqr(k, lane, a, d); break;
    case CQ_OP_CYC: cq_cyc_sqr(k, lane, a, d); break;
    case CQ_OP_COPY: cq_copy(k, lane, a, d); break;
    case CQ_OP_CONJ: cq_conj(k, lane, a, d); break;
    case CQ_OP_FROB1: cq_frob<1>(k, lane, a, d); break;
    case CQ_OP_FROB2: cq_frob<2>(k, lane, a, d); break;
    case CQ_OP_INV6: cq_inv6(k, lane, a, d); break;
    default: break;
  }
}

// Final exponentiation program (arkworks exponent: easy part, then (x-1)^2 (x+p)(x^2+p^2-1) + 3).
// Input in buffer 0, result in buffer CQ_FE_OUT; 5 buffers.  Returns the number of ops written (<= CQ_FE_MAXOPS).
constexpr int CQ_FE_NBUF = 5, CQ_FE_OUT = 3, CQ_FE_MAXOPS = 400;
inline int cq_build_final_exp(uint32_t* prog) {
  int n = 0;
  auto I = [&](int op, int dst, int a, int b = 0) { prog[n++] = cq_ins(op, dst, a, b); };
  // dst = src^|x| conjugated, via the ping-pong buffers 0/1 (src must not be 0 or 1)
  auto exp_x = [&](int dst, int src) {
    I(CQ_OP_COPY, 0, src);
    int cur = 0;
    for (int bit = 62; bit >= 0; bit--) {
      I(CQ_OP_CYC, cur ^ 1, cur);
      cur ^= 1;
      if ((0xd201000000010000ull >> bit) & 1) {
        I(CQ_OP_MUL, cur ^ 1, cur, src);
        cur ^= 1;
      }
    }
    I(CQ_OP_CONJ, dst, cur);
  };
  // easy part: r = f^((p^6-1)(p^2+1)) = frob2(g) * g,  g = conj(f)^2 / (f conj(f))
  I(CQ_OP_CONJ, 1, 0);
  I(CQ_OP_MUL, 2, 0, 1);   // N = f * conj(f)  in Fp6
  I(CQ_OP_INV6, 2, 2);
  I(CQ_OP_SQR, 3, 1);
  I(CQ_OP_MUL, 0, 3, 2);   // g
  I(CQ_OP_FROB2, 1, 0);
  I(CQ_OP_MUL, 4, 1, 0);   // r  (kept in 4)
  // a = r^(x-1)
  exp_x(2, 4);
  I(CQ_OP_CONJ, 1, 4);
  I(CQ_OP_MUL, 3, 2, 1);   // a in 3
  // b = a^(x-1)
  exp_x(2, 3);
  I(CQ_OP_CONJ, 1, 3);
  I(CQ_OP_MUL, 3, 2, 1);   // b in 3  (a dead)
  // c = b^(x+p)
  exp_x(2, 3);
  I(CQ_OP_FROB1, 1, 3);
  I(CQ_OP_MUL, 3, 2, 1);   // c in 3
  // d = c^(x^2) * c^(p^2) * conj(c)
  exp_x(2, 3);
  exp_x(2, 2);             // copies 2 -> 0 first, so in == out is fine
  I(CQ_OP_FROB2, 1, 3);
  I(CQ_OP_MUL, 0, 2, 1);
  I(CQ_OP_CONJ, 1, 3);
  I(CQ_OP_MUL, 2, 0, 1);   // d in 2
  // r^3
  I(CQ_OP_CYC, 0, 4);
  I(CQ_OP_MUL, 1, 0, 4);
  I(CQ_OP_MUL, 3, 2, 1);   // result in 3
  return n;
}

// ------------------------------------------------------------------ block shape
// A thread block holds CQ_GROUPS independent 6-warp groups (12 warps = 3 per SM sub-partition, so the four
// schedulers of an SM carry the same load: with 6-warp blocks two of them get two warps of every block and
// the group barrier makes everyone wait for those).  Each group synchronises on its own named barrier.
constexpr int CQ_GROUPS = 2;
constexpr int CQ_GROUP_THREADS = 6 * CQ_LANES;
constexpr int CQ_BLOCK_THREADS = CQ_GROUPS * CQ_GROUP_THREADS;
#if defined(__CUDACC__)
__device__ GS_INL void cq_group_sync(int group) {
  asm volatile("bar.sync %0, %1;" ::"r"(group + 1), "r"(CQ_GROUP_THREADS) : "memory");
}
#endif

// ------------------------------------------------------------------ constants / conversion
GS_HD GS_INL void cq_set_one(int k, int lane, uint32_t* f) {
  fp2 r;
  r.set_zero();
  if (k == 0) fp_one(r.c0);
  cq_st_coef(f, k, lane, r);
}
// position (in Fp2 units) of w-basis coefficient k inside the tower-ordered fp12
GS_HD GS_INL int cq_tower_pos(int k) { return (k & 1) * 3 + (k >> 1); }

}  // namespace gs
