// BLS12-381 base field Fp (12 x 32-bit limbs) and scalar field Fr (8 x 32-bit limbs),
// Montgomery form with R = 2^384 / 2^256 -- bit-identical to arkworks' 6x64 / 4x64
// in-memory representation (SURVEY.md §8b), so no conversion happens at the C ABI.
//
// Replaces (reference call sites): every ark-ff field operation underneath
// src/data_structures.rs:336-342, 484-502, 768-913.
//
// Device path: IMAD.WIDE.U32(.X) carry chains (mad.lo.cc / madc.hi.cc pairs that ptxas
// fuses into one wide multiply-add), operands in registers, modulus limbs as immediates.
// Host path (`GS_HOST_SIM`, tests only): the SAME limb algorithm with the PTX carry
// primitives emulated in C so the device formulas can be checked on a CPU-only box.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define GS_HD __host__ __device__
#define GS_INL __forceinline__
#else
#define GS_HD
#define GS_INL inline __attribute__((always_inline))
#endif
#if defined(__CUDA_ARCH__)
#define GS_NOINL __noinline__
#else
#define GS_NOINL
#endif

namespace gs {

// ------------------------------------------------------------------ carry-chain primitives
#if defined(__CUDA_ARCH__)
#define GS_PTX3(name, ins)                                                                   \
  __device__ GS_INL uint32_t name(uint32_t a, uint32_t b) {                                  \
    uint32_t r; asm volatile(ins " %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
#define GS_PTX4(name, ins)                                                                   \
  __device__ GS_INL uint32_t name(uint32_t a, uint32_t b, uint32_t c) {                      \
    uint32_t r; asm volatile(ins " %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(c)); return r; }
GS_PTX3(add_cc, "add.cc.u32")
GS_PTX3(addc_cc, "addc.cc.u32")
GS_PTX3(addc, "addc.u32")
GS_PTX3(sub_cc, "sub.cc.u32")
GS_PTX3(subc_cc, "subc.cc.u32")
GS_PTX3(subc, "subc.u32")
GS_PTX4(mad_lo_cc, "mad.lo.cc.u32")
GS_PTX4(madc_lo_cc, "madc.lo.cc.u32")
GS_PTX4(mad_hi_cc, "mad.hi.cc.u32")
GS_PTX4(madc_hi_cc, "madc.hi.cc.u32")
GS_PTX4(madc_hi, "madc.hi.u32")
__device__ GS_INL uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
__device__ GS_INL uint32_t mul_hi(uint32_t a, uint32_t b) { return __umulhi(a, b); }
// full 32x32 -> 64 product as ONE IMAD.WIDE (lo, hi land in a register pair)
__device__ GS_INL void mul_wide(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
  asm volatile("{\n\t.reg .u64 t;\n\tmul.wide.u32 t, %2, %3;\n\tmov.b64 {%0, %1}, t;\n\t}" : "=r"(lo), "=r"(hi) : "r"(a), "r"(b));
}
#else
// host emulation of the PTX condition-code register (tests only)
static thread_local uint32_t g_cc = 0;
GS_INL uint32_t add_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b; g_cc = (uint32_t)(t >> 32); return (uint32_t)t; }
GS_INL uint32_t addc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b + g_cc; g_cc = (uint32_t)(t >> 32); return (uint32_t)t; }
GS_INL uint32_t addc(uint32_t a, uint32_t b) { return a + b + g_cc; }
GS_INL uint32_t sub_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b; g_cc = (uint32_t)(t >> 63); return (uint32_t)t; }
GS_INL uint32_t subc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b - g_cc; g_cc = (uint32_t)(t >> 63); return (uint32_t)t; }
GS_INL uint32_t subc(uint32_t a, uint32_t b) { return a - b - g_cc; }
GS_INL uint32_t mul_lo(uint32_t a, uint32_t b) { return a * b; }
GS_INL uint32_t mul_hi(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
GS_INL void mul_wide(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a * b; lo = (uint32_t)t; hi = (uint32_t)(t >> 32); }
GS_INL uint32_t mad_lo_cc(uint32_t a, uint32_t b, uint32_t c) { return add_cc(mul_lo(a, b), c); }
GS_INL uint32_t madc_lo_cc(uint32_t a, uint32_t b, uint32_t c) { return addc_cc(mul_lo(a, b), c); }
GS_INL uint32_t mad_hi_cc(uint32_t a, uint32_t b, uint32_t c) { return add_cc(mul_hi(a, b), c); }
GS_INL uint32_t madc_hi_cc(uint32_t a, uint32_t b, uint32_t c) { return addc_cc(mul_hi(a, b), c); }
GS_INL uint32_t madc_hi(uint32_t a, uint32_t b, uint32_t c) { return addc(mul_hi(a, b), c); }
#endif

// ------------------------------------------------------------------ field parameters
struct FpParams {
  static constexpr int N = 12;
  static constexpr uint32_t M0 = 0xfffcfffdu;  // -p^-1 mod 2^32
  GS_HD static constexpr uint32_t mod(int i) {
    constexpr uint32_t t[12] = {0xffffaaabu, 0xb9feffffu, 0xb153ffffu, 0x1eabfffeu, 0xf6b0f624u, 0x6730d2a0u,
                                0xf38512bfu, 0x64774b84u, 0x434bacd7u, 0x4b1ba7b6u, 0x397fe69au, 0x1a0111eau};
    return t[i];
  }
};
struct FrParams {
  static constexpr int N = 8;
  static constexpr uint32_t M0 = 0xffffffffu;  // -r^-1 mod 2^32
  GS_HD static constexpr uint32_t mod(int i) {
    constexpr uint32_t t[8] = {0x00000001u, 0xffffffffu, 0xfffe5bfeu, 0x53bda402u,
                               0x09a1d805u, 0x3339d808u, 0x299d7d48u, 0x73eda753u};
    return t[i];
  }
};

// ------------------------------------------------------------------ generic Montgomery kernel code
template <class PR>
struct Mont {
  static constexpr int N = PR::N;
  uint32_t l[N];

  // r = a + b mod p   (inputs < p)
  GS_HD static GS_INL void add(Mont& r, const Mont& a, const Mont& b) {
    uint32_t t[N], s[N];
    t[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = addc_cc(a.l[i], b.l[i]);
    t[N - 1] = addc(a.l[N - 1], b.l[N - 1]);  // p < 2^(32N-1): no carry out
    s[0] = sub_cc(t[0], PR::mod(0));
#pragma unroll
    for (int i = 1; i < N; i++) s[i] = subc_cc(t[i], PR::mod(i));
    uint32_t borrow = subc(0u, 0u);  // 0xffffffff if t < p
#pragma unroll
    for (int i = 0; i < N; i++) r.l[i] = borrow ? t[i] : s[i];
  }

  // r = a - b mod p
  GS_HD static GS_INL void sub(Mont& r, const Mont& a, const Mont& b) {
    uint32_t t[N];
    t[0] = sub_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < N; i++) t[i] = subc_cc(a.l[i], b.l[i]);
    uint32_t mask = subc(0u, 0u);  // all-ones if borrow
    r.l[0] = add_cc(t[0], PR::mod(0) & mask);
#pragma unroll
    for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(t[i], PR::mod(i) & mask);
    r.l[N - 1] = addc(t[N - 1], PR::mod(N - 1) & mask);
  }

  GS_HD static GS_INL void neg(Mont& r, const Mont& a) {
    uint32_t nz = 0;
#pragma unroll
    for (int i = 0; i < N; i++) nz |= a.l[i];
    uint32_t mask = nz ? 0xffffffffu : 0u;
    uint32_t t[N];
    t[0] = sub_cc(PR::mod(0), a.l[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = subc_cc(PR::mod(i), a.l[i]);
    t[N - 1] = subc(PR::mod(N - 1), a.l[N - 1]);
#pragma unroll
    for (int i = 0; i < N; i++) r.l[i] = t[i] & mask;
  }

  GS_HD static GS_INL void dbl(Mont& r, const Mont& a) { add(r, a, a); }

  GS_HD GS_INL bool is_zero() const {
    uint32_t nz = 0;
#pragma unroll
    for (int i = 0; i < N; i++) nz |= l[i];
    return nz == 0;
  }
  GS_HD GS_INL bool equals(const Mont& o) const {
    uint32_t d = 0;
#pragma unroll
    for (int i = 0; i < N; i++) d |= l[i] ^ o.l[i];
    return d == 0;
  }
  GS_HD GS_INL void set_zero() {
#pragma unroll
    for (int i = 0; i < N; i++) l[i] = 0;
  }

  // ---- Montgomery product, even/odd accumulator formulation.
  // T is held as  sum E[k] W^k + sum O[k] W^(k+1)  so that every 64-bit partial product
  // (lo,hi) lands in an adjacent register pair of ONE array and each row is two carry
  // chains of N/2 fused IMAD.WIDE.U32.X; the per-row right shift is free (it is folded
  // into the addend operand of the next row, see `row`).
  //   acc[j], acc[j+1] += x[j] * y   for j = 0,2,..,N-2, one carry chain, carry left in CC
  GS_HD static GS_INL void cmad_row(uint32_t* acc, const uint32_t* x, uint32_t y) {
    acc[0] = mad_lo_cc(x[0], y, acc[0]);
    acc[1] = madc_hi_cc(x[0], y, acc[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      acc[j] = madc_lo_cc(x[j], y, acc[j]);
      acc[j + 1] = madc_hi_cc(x[j], y, acc[j + 1]);
    }
  }
  // same with the modulus (limbs become immediates); off = 0 (even limbs) or 1 (odd limbs)
  template <int OFF>
  GS_HD static GS_INL void cmad_row_mod(uint32_t* acc, uint32_t y) {
    acc[0] = mad_lo_cc(PR::mod(OFF), y, acc[0]);
    acc[1] = madc_hi_cc(PR::mod(OFF), y, acc[1]);
#pragma unroll
    for (int j = 2; j < N; j += 2) {
      acc[j] = madc_lo_cc(PR::mod(j + OFF), y, acc[j]);
      acc[j + 1] = madc_hi_cc(PR::mod(j + OFF), y, acc[j + 1]);
    }
  }
  //   acc[j], acc[j+1] = x[j] * y + acc[j+2], acc[j+3]   (consumes the CC left by the caller)
  GS_HD static GS_INL void madc_row_rshift(uint32_t* acc, const uint32_t* x, uint32_t y) {
#pragma unroll
    for (int j = 0; j < N - 2; j += 2) {
      acc[j] = madc_lo_cc(x[j], y, acc[j + 2]);
      acc[j + 1] = madc_hi_cc(x[j], y, acc[j + 3]);
    }
    acc[N - 2] = madc_lo_cc(x[N - 2], y, 0u);
    acc[N - 1] = madc_hi(x[N - 2], y, 0u);
  }
  // one CIOS row:  T += a*bi ; m = T0 * M0 ; T += m*p ; T >>= 32   (E/O swap roles each row)
  GS_HD static GS_INL void row(uint32_t* E, uint32_t* O, const uint32_t* a, uint32_t bi, bool first) {
    if (first) {
#pragma unroll
      for (int j = 0; j < N; j += 2) {
        mul_wide(E[j], E[j + 1], a[j], bi);
        mul_wide(O[j], O[j + 1], a[j + 1], bi);
      }
    } else {
      // here E is last row's O (already at the right position) and O is last row's E,
      // which sits two words too high: O[1] belongs to position 0, O[k+2] to O-slot k.
      E[0] = add_cc(E[0], O[1]);
      madc_row_rshift(O, a + 1, bi);
      cmad_row(E, a, bi);
      O[N - 1] = addc(O[N - 1], 0u);
    }
    uint32_t m = mul_lo(E[0], PR::M0);
    cmad_row_mod<1>(O, m);
    cmad_row_mod<0>(E, m);
    O[N - 1] = addc(O[N - 1], 0u);
  }

  GS_HD static GS_INL void final_sub(Mont& r, const uint32_t* t) {
    uint32_t s[N];
    s[0] = sub_cc(t[0], PR::mod(0));
#pragma unroll
    for (int i = 1; i < N; i++) s[i] = subc_cc(t[i], PR::mod(i));
    uint32_t borrow = subc(0u, 0u);
#pragma unroll
    for (int i = 0; i < N; i++) r.l[i] = borrow ? t[i] : s[i];
  }

  GS_HD static GS_INL void mul(Mont& r, const Mont& a, const Mont& b) {
    // Operands are copied into locals first: when a / b are references into memory (out-of-line callers,
    // possible aliasing with r) ptxas otherwise fails to fuse the mad.lo.cc / madc.hi.cc pairs of the a*b rows
    // into IMAD.WIDE.U32.X and emits IMAD + IMAD.HI + 2 IADD3.X per limb product instead (measured: 144
    // unfused pairs per product, 2.4x the instructions).
    uint32_t E[N], O[N], al[N], bl[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
      al[i] = a.l[i];
      bl[i] = b.l[i];
    }
#pragma unroll
    for (int i = 0; i < N; i += 2) {
      row(E, O, al, bl[i], i == 0);
      row(O, E, al, bl[i + 1], false);
    }
    // after an even number of rows the roles are swapped back: T = sum O[k] W^k + sum E[k] W^(k+1)
    // result = T / W = (O >> 32) + E
    uint32_t t[N];
    t[0] = add_cc(O[1], E[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = addc_cc(O[i + 1], E[i]);
    t[N - 1] = addc(0u, E[N - 1]);
    final_sub(r, t);
  }
  GS_HD static GS_INL void sqr(Mont& r, const Mont& a) { mul(r, a, a); }

  // ---- sum of products with ONE interleaved Montgomery reduction ("lazy reduction"):
  //     r = (a[0] b[0] + ... + a[NT-1] b[NT-1]) / R  mod p
  // Every CIOS row adds the NT partial-product rows first and then a single m*p row, i.e.
  // NT*N*N + N*N + N multiply-adds instead of NT*(2*N*N + N).  `units` = sum over the terms of
  // (bound of a[t] / p) * (bound of b[t] / p) (1 for canonical inputs; operands that are plain sums
  // of two canonical values count 2).  Requires (units + 1) * p < 2^(32N): the running value stays
  // below that, and the final value is < (units * p / R + 1) * p < 2p, so one conditional
  // subtraction canonicalises it.  For BLS12-381 Fp (R/p = 9.84): units <= 8.
  template <int NT>
  GS_HD static GS_INL void mulsum(Mont& r, const Mont (&a)[NT], const Mont (&b)[NT]) {
    uint32_t E[N], O[N];
#pragma unroll
    for (int i = 0; i < N; i += 2) {
      rowsum<NT>(E, O, a, b, i, i == 0);
      rowsum<NT>(O, E, a, b, i + 1, false);
    }
    uint32_t t[N];
    t[0] = add_cc(O[1], E[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = addc_cc(O[i + 1], E[i]);
    t[N - 1] = addc(0u, E[N - 1]);
    final_sub(r, t);
  }
  template <int NT>
  GS_HD static GS_INL void rowsum(uint32_t* E, uint32_t* O, const Mont (&a)[NT], const Mont (&b)[NT], int i, bool first) {
    if (first) {
#pragma unroll
      for (int j = 0; j < N; j += 2) {
        mul_wide(E[j], E[j + 1], a[0].l[j], b[0].l[i]);
        mul_wide(O[j], O[j + 1], a[0].l[j + 1], b[0].l[i]);
      }
    } else {
      E[0] = add_cc(E[0], O[1]);
      madc_row_rshift(O, a[0].l + 1, b[0].l[i]);
      cmad_row(E, a[0].l, b[0].l[i]);
      O[N - 1] = addc(O[N - 1], 0u);
    }
#pragma unroll
    for (int t = 1; t < NT; t++) {
      cmad_row(O, a[t].l + 1, b[t].l[i]);  // no carry out of the window: the value is < 2^(32(N+1))
      cmad_row(E, a[t].l, b[t].l[i]);
      O[N - 1] = addc(O[N - 1], 0u);
    }
    uint32_t m = mul_lo(E[0], PR::M0);
    cmad_row_mod<1>(O, m);
    cmad_row_mod<0>(E, m);
    O[N - 1] = addc(O[N - 1], 0u);
  }
  // ---- the same interleaved sum of products with the b-side limbs supplied row by row (`bl[t]` = limb i of
  // b[t]), so that the b operands can be streamed out of shared memory a quad at a time instead of being
  // held in registers (coop12.cuh).  Row i uses rowsum_l(E, O, ...) for even i and rowsum_l(O, E, ...) for odd i;
  // after the N rows mulsum_finish() produces the canonical value.
  template <int NT>
  GS_HD static GS_INL void rowsum_l(uint32_t* E, uint32_t* O, const Mont (&a)[NT], const uint32_t (&bl)[NT], bool first) {
    if (first) {
#pragma unroll
      for (int j = 0; j < N; j += 2) {
        mul_wide(E[j], E[j + 1], a[0].l[j], bl[0]);
        mul_wide(O[j], O[j + 1], a[0].l[j + 1], bl[0]);
      }
    } else {
      E[0] = add_cc(E[0], O[1]);
      madc_row_rshift(O, a[0].l + 1, bl[0]);
      cmad_row(E, a[0].l, bl[0]);
      O[N - 1] = addc(O[N - 1], 0u);
    }
#pragma unroll
    for (int t = 1; t < NT; t++) {
      cmad_row(O, a[t].l + 1, bl[t]);
      cmad_row(E, a[t].l, bl[t]);
      O[N - 1] = addc(O[N - 1], 0u);
    }
    uint32_t m = mul_lo(E[0], PR::M0);
    cmad_row_mod<1>(O, m);
    cmad_row_mod<0>(E, m);
    O[N - 1] = addc(O[N - 1], 0u);
  }
  GS_HD static GS_INL void mulsum_finish(Mont& r, const uint32_t* E, const uint32_t* O) {
    uint32_t t[N];
    window_out(t, E, O);
    final_sub(r, t);
  }
  // the window after an even number of rows, divided by W: t = (O >> 32) + E
  GS_HD static GS_INL void window_out(uint32_t* t, const uint32_t* E, const uint32_t* O) {
    t[0] = add_cc(O[1], E[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = addc_cc(O[i + 1], E[i]);
    t[N - 1] = addc(0u, E[N - 1]);
  }

  // ---- the rows of rowsum_l WITHOUT the reduction: P = sum_t a[t] b[t] as an unreduced 2N-limb integer ("wide"), so
  // that several such sums can be combined before ONE reduction (coop12.cuh cq_fp2_dot_w).  After row i, [0] of the
  // E argument is limb i of P: it leaves the window (the next row never reads that slot).  After the N rows
  // window_out(hi, E, O) gives limbs N..2N-1.  The window holds floor(partial sum / W^i) < (sum_t a[t]) W, so it fits
  // N + 1 limbs (no carry out of O[N-1]) when sum_t a[t] < R; the b[t] may be anything below R.
  template <int NT>
  GS_HD static GS_INL void rowsum_w(uint32_t* E, uint32_t* O, const Mont (&a)[NT], const uint32_t (&bl)[NT], bool first) {
    if (first) {
#pragma unroll
      for (int j = 0; j < N; j += 2) {
        mul_wide(E[j], E[j + 1], a[0].l[j], bl[0]);
        mul_wide(O[j], O[j + 1], a[0].l[j + 1], bl[0]);
      }
    } else {
      E[0] = add_cc(E[0], O[1]);
      madc_row_rshift(O, a[0].l + 1, bl[0]);
      cmad_row(E, a[0].l, bl[0]);
      O[N - 1] = addc(O[N - 1], 0u);
    }
#pragma unroll
    for (int t = 1; t < NT; t++) {
      cmad_row(O, a[t].l + 1, bl[t]);
      cmad_row(E, a[t].l, bl[t]);
      O[N - 1] = addc(O[N - 1], 0u);
    }
  }
  // ---- one Montgomery reduction of a wide value:  r = (lo + hi R) / R mod p,  for lo + hi R < p R.
  // The rows of `row` without the a*b part take the window from lo to t = (lo + M p) / R <= p (M < R the Montgomery
  // quotient; the window stays below R / W^i + p + 1 < 2^(32(N+1))).  hi <= p - 1, so t + hi < 2p and one
  // conditional subtraction canonicalises it.  N*N + N multiply-adds, like the reduction part of mulsum.
  GS_HD static GS_INL void redc_w(Mont& r, const uint32_t (&lo)[N], const uint32_t (&hi)[N]) {
    uint32_t E[N], O[N];
#pragma unroll
    for (int i = 0; i < N; i++) {
      E[i] = lo[i];
      O[i] = 0u;
    }
#pragma unroll
    for (int i = 0; i < N; i += 2) {
      redc_row(E, O, i == 0);
      redc_row(O, E, false);
    }
    uint32_t t[N];
    window_out(t, E, O);
    t[0] = add_cc(t[0], hi[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) t[i] = addc_cc(t[i], hi[i]);
    t[N - 1] = addc(t[N - 1], hi[N - 1]);
    final_sub(r, t);
  }
  GS_HD static GS_INL void redc_row(uint32_t* E, uint32_t* O, bool first) {
    uint32_t m;
    if (first) {
      m = mul_lo(E[0], PR::M0);
      cmad_row_mod<1>(O, m);
    } else {
      // as in `row`: E is last row's O, O is last row's E two slots too high (O[1] at position 0); the carry of the
      // position-0 merge goes into the shifted O chain
      E[0] = add_cc(E[0], O[1]);
      m = mul_lo(E[0], PR::M0);
#pragma unroll
      for (int j = 0; j < N - 2; j += 2) {
        O[j] = madc_lo_cc(PR::mod(j + 1), m, O[j + 2]);
        O[j + 1] = madc_hi_cc(PR::mod(j + 1), m, O[j + 3]);
      }
      O[N - 2] = madc_lo_cc(PR::mod(N - 1), m, 0u);
      O[N - 1] = madc_hi(PR::mod(N - 1), m, 0u);
    }
    cmad_row_mod<0>(E, m);
    O[N - 1] = addc(O[N - 1], 0u);
  }
  // plain limb-wise sum without reduction (inputs < p, result < 2p): an operand for mulsum that counts 2 units
  GS_HD static GS_INL void add_noreduce(Mont& r, const Mont& a, const Mont& b) {
    r.l[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < N - 1; i++) r.l[i] = addc_cc(a.l[i], b.l[i]);
    r.l[N - 1] = addc(a.l[N - 1], b.l[N - 1]);
  }
};

typedef Mont<FpParams> fp;
typedef Mont<FrParams> fr;

}  // namespace gs
