// Extraction with the binding key (gs_extract, extract.cu): X = c.1 - a c.0 for a commitment c made under
// u = [(p1, a p1), t (p1, a p1)] (likewise on G2), as host/device functions so that tests/hostsim runs the same code on the
// CPU.  The key a is the same for every element of a call: it is split along the endomorphism and recoded into signed
// 4-bit windows ONCE on the host, and the digits are a kernel parameter, so every lane runs the same instruction stream.
//   G1:  a = k1 + k2 x^2 (glv_split),  a P = k1 P + k2 (-phi(P)),  k1, k2 < 2^128:  33 positions x 2 parts
//   G2:  a = sum_j c_j |x|^j (gls_split),  a Q = sum_j c_j (-1)^j psi^j(Q),  c_j < 2^64:  17 positions x 4 parts
// One Straus walk per element: the parts share the doublings (128 on G1, 64 on G2), and the parts' table entries are the
// endomorphism images of one table 1P .. 8P.
#pragma once
#include <cstring>

#include "endo.cuh"

namespace gs {

struct extract_digits {
  int8_t d[4][33];  // d[part][position] in [-8, 8), least significant position first
  int npos;         // positions up to the highest non-zero digit of any part (0: the key is 0)
};

template <class F>
struct ExtractEndo;
template <>
struct ExtractEndo<FpOps> {
  static constexpr int PARTS = 2, WINDOWS = 32;  // 128-bit halves
  // e <- the part-j image of e: -phi(e) = (beta X, -Y, Z) for j = 1
  GS_HD static GS_INL void image(g1_jac& e, int j) {
    if (j == 0) return;
    endo_phi_x(e.X, e.X);
    fp::neg(e.Y, e.Y);
  }
};
// psi in Jacobian coordinates: x = X / Z^2 gives psi(x) = conj(X) cx / conj(Z)^2, so (conj(X) cx, conj(Y) cy, conj(Z))
static GS_HD GS_NOINL void endo_psi_jac(g2_jac& e) {
  fp c1;
  fp2 cy, t;
#pragma unroll
  for (int j = 0; j < 12; j++) {
    c1.l[j] = GS_ENDO_AT(PSI_CX_C1, j);
    cy.c0.l[j] = GS_ENDO_AT(PSI_CY_C0, j);
    cy.c1.l[j] = GS_ENDO_AT(PSI_CY_C1, j);
  }
  fp a, b;  // conj(X) * (c1 u) = X.c1 c1 + X.c0 c1 u
  fp::mul(a, e.X.c1, c1);
  fp::mul(b, e.X.c0, c1);
  e.X.c0 = a;
  e.X.c1 = b;
  fp2::conj(t, e.Y);
  fp2::mul(e.Y, t, cy);
  fp2::conj(e.Z, e.Z);
}
template <>
struct ExtractEndo<Fp2Ops> {
  static constexpr int PARTS = 4, WINDOWS = 16;  // 64-bit digits in base |x|
  // e <- (-1)^j psi^j(e)
  GS_HD static GS_INL void image(g2_jac& e, int j) {
#pragma unroll 1
    for (int i = 0; i < j; i++) endo_psi_jac(e);
    if (j & 1) fp2::neg(e.Y, e.Y);
  }
};

// signed 4-bit windows of the low 4 * nwin bits of k, and the carry out of the top window at position nwin
static inline void extract_recode(int8_t* d, const uint32_t* k, int nwin) {
  int carry = 0;
  for (int i = 0; i < nwin; i++) {
    int v = (int)((k[i >> 3] >> ((i & 7) * 4)) & 15u) + carry;
    carry = v >= 8;
    d[i] = (int8_t)(carry ? v - 16 : v);
  }
  d[nwin] = (int8_t)carry;
}

// the digits of the key a (canonical limbs, < r); host side, once per call
template <class F>
static inline extract_digits make_extract_digits(const uint32_t k[8]);
template <>
inline extract_digits make_extract_digits<FpOps>(const uint32_t k[8]) {
  extract_digits r;
  memset(&r, 0, sizeof r);
  uint32_t k1[4], k2[4];
  glv_split(k1, k2, k);
  extract_recode(r.d[0], k1, 32);
  extract_recode(r.d[1], k2, 32);
  for (int i = 0; i <= 32; i++)
    if (r.d[0][i] || r.d[1][i]) r.npos = i + 1;
  return r;
}
template <>
inline extract_digits make_extract_digits<Fp2Ops>(const uint32_t k[8]) {
  extract_digits r;
  memset(&r, 0, sizeof r);
  uint64_t c[4];
  gls_split(c, k);
  for (int j = 0; j < 4; j++) {
    const uint32_t kk[2] = {(uint32_t)c[j], (uint32_t)(c[j] >> 32)};
    extract_recode(r.d[j], kk, 16);
  }
  for (int i = 0; i <= 16; i++)
    if (r.d[0][i] || r.d[1][i] || r.d[2][i] || r.d[3][i]) r.npos = i + 1;
  return r;
}

// tab[i] = (i + 1) P, Jacobian (all identities when P is)
template <class F>
GS_HD GS_INL void extract_table(Jac<F> (&tab)[8], const Aff<F>& p) {
  tab[0].from_affine(p);
  Jac<F>::dbl(tab[1], tab[0]);
#pragma unroll 1
  for (int i = 2; i < 8; i++) Jac<F>::add_mixed(tab[i], tab[i - 1], p);
}

// acc = a P from the table of P: one walk, four shared doublings per position, one addition per non-zero digit
template <class F>
GS_HD GS_INL void extract_walk(Jac<F>& acc, const Jac<F> (&tab)[8], const extract_digits& dg) {
  acc.set_inf();
#pragma unroll 1
  for (int i = dg.npos - 1; i >= 0; i--) {
    if (i != dg.npos - 1) {
      Jac<F>::dbl(acc, acc);
      Jac<F>::dbl(acc, acc);
      Jac<F>::dbl(acc, acc);
      Jac<F>::dbl(acc, acc);
    }
#pragma unroll 1
    for (int j = 0; j < ExtractEndo<F>::PARTS; j++) {
      const int d = dg.d[j][i];
      if (d == 0) continue;
      Jac<F> e = tab[(d < 0 ? -d : d) - 1];
      ExtractEndo<F>::image(e, j);
      if (d < 0) F::neg(e.Y, e.Y);
      Jac<F>::add(acc, acc, e);
    }
  }
}

// acc = c.1 - a c.0, not yet normalised (the kernel normalises a block at once)
template <class F>
GS_HD GS_INL void extract_jac(Jac<F>& acc, const Aff<F>& c0, const Aff<F>& c1, const extract_digits& dg) {
  Jac<F> tab[8];
  extract_table<F>(tab, c0);
  extract_walk<F>(acc, tab, dg);
  Jac<F>::neg(acc, acc);
  Jac<F>::add_mixed(acc, acc, c1);
}

// one element in one thread (tests)
template <class F>
GS_HD GS_INL void extract_single(Aff<F>& out, const Aff<F>& c0, const Aff<F>& c1, const extract_digits& dg) {
  Jac<F> acc;
  extract_jac<F>(acc, c0, c1, dg);
  Jac<F>::to_affine(out, acc);
}

}  // namespace gs
