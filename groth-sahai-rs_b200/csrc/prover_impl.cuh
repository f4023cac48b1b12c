// Prover-side kernels templated over the group (F = FpOps: G1, F = Fp2Ops: G2) and their host drivers.
// Instantiated once per group in prover_g1.cu / prover_g2.cu so the two halves compile in parallel.
// Reference: src/prover/commit.rs:78-256, src/prover/prove.rs:92-488, src/data_structures.rs:645-742.
#pragma once
#include "batchinv.cuh"
#include "ctx.h"
#include "endo.cuh"

namespace gs {

// ------------------------------------------------------------------ fixed-base window tables
// For base point B (one coordinate of u1, u2, W1 / v1, v2, W2) and window w:
//     T[w][d-1] = d * 2^(c w) * B,   d = 1 .. 2^(c-1)     (signed digits => half tables)
// layout: tab[((base*2 + a) * W + w) * H + (d-1)]
constexpr int GS_TAB_NT = 128;
#ifndef GS_FC_G2_BLOCKS
#define GS_FC_G2_BLOCKS 2
#endif

template <class F>
__global__ void k_table_window_bases(const Aff<F>* __restrict__ bases, Aff<F>* __restrict__ tab, int c, int W, size_t H) {
  // one thread per base point: writes d = 1 entries (2^(cw) B) for every window
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= 6) return;
  Jac<F> j;
  j.from_affine(bases[b]);
  for (int w = 0; w < W; w++) {
    Aff<F> a;
    Jac<F>::to_affine(a, j);
    tab[((size_t)b * W + w) * H] = a;
    for (int i = 0; i < c; i++) Jac<F>::dbl(j, j);
  }
}

// thread -> (base b, window w, run r): entries d = r*RUN+1 .. r*RUN+RUN of T[b][w] by a chain of
// mixed additions from a small scalar-mul start, normalised with a block-wide batch inversion per step.
template <class F, int RUN>
__global__ void __launch_bounds__(GS_TAB_NT) k_table_fill(Aff<F>* __restrict__ tab, int W, size_t H) {
  __shared__ fp sm[2 * GS_TAB_NT];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t runs_per_row = (H + RUN - 1) / RUN;
  size_t total = (size_t)6 * W * runs_per_row;
  bool active = id < total;
  size_t row = active ? id / runs_per_row : 0, r = active ? id % runs_per_row : 0;
  Aff<F>* T = tab + row * H;
  Aff<F> B = T[0];
  Jac<F> acc;
  uint32_t k[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  k[0] = (uint32_t)(r * RUN);  // start = (r*RUN) * B
  scalar_mul<F>(acc, B, k);
  for (int i = 0; i < RUN; i++) {
    Jac<F>::add_mixed(acc, acc, B);
    Aff<F> a;
    block_to_affine<GS_TAB_NT>(a, acc, sm);
    size_t d1 = r * RUN + i;  // d - 1
    if (active && d1 < H && d1 > 0) T[d1] = a;
  }
}

// ------------------------------------------------------------------ batch commitments
// out[i].p[a] = s0_i * Base0.a + s1_i * Base1.a  (+ addend_i when a == 1)
//   batch_commit_G1 (commit.rs:78-100):            s0,s1 = R[i][0], R[i][1]; bases u1,u2; addend X_i
//   batch_commit_scalar_to_B1 (commit.rs:125-156): s0 = x_i, s1 = r_i;     bases W1,u1; no addend
// thread -> (i, a); signed c-bit windows; one table lookup + one mixed addition per window.
// c bits of the 256-bit integer k starting at `bit` (zero beyond bit 255); c <= 16
GS_HD GS_INL uint32_t get_bits(const uint32_t k[8], int bit, int c) {
  int w = bit >> 5, s = bit & 31;
  if (w >= 8) return 0;
  uint64_t v = k[w];
  if (w + 1 < 8) v |= (uint64_t)k[w + 1] << 32;
  return (uint32_t)(v >> s) & ((1u << c) - 1u);
}

template <class F>
GS_HD GS_INL void fixed_base_accumulate(Jac<F>& acc, const Aff<F>* __restrict__ T /* [W][H] */, const uint32_t k[8], int c,
                                        int W, size_t H) {
  // digits recoded into (-2^(c-1), 2^(c-1)]; the table entry of window w + 1 is fetched before the (out-of-line)
  // addition of window w runs, so the dependent load never stalls in front of its own addition
  uint32_t carry = 0;
  const uint32_t half = 1u << (c - 1);
  Aff<F> cur, nxt;
  bool cur_nz = false, cur_neg = false, nxt_nz = false, nxt_neg = false;
  auto fetch = [&](int w, Aff<F>& e, bool& nz, bool& ng) {
    uint32_t d = get_bits(k, w * c, c) + carry;
    ng = d > half;
    carry = ng ? 1u : 0u;
    uint32_t mag = ng ? (1u << c) - d : d;
    nz = mag != 0;
    if (nz) e = T[(size_t)w * H + (mag - 1)];
  };
  fetch(0, cur, cur_nz, cur_neg);
  for (int w = 0; w < W; w++) {
    nxt_nz = false;
    if (w + 1 < W) fetch(w + 1, nxt, nxt_nz, nxt_neg);
    if (cur_nz) {
      if (cur_neg) F::neg(cur.y, cur.y);
      Jac<F>::add_mixed(acc, acc, cur);
    }
    cur = nxt;
    cur_nz = nxt_nz;
    cur_neg = nxt_neg;
  }
}

// the windows [w0, w1) only (the recoding carry of the lower windows is recomputed: integer work, no curve operation)
template <class F>
GS_HD GS_INL void fixed_base_accumulate_range(Jac<F>& acc, const Aff<F>* __restrict__ T, const uint32_t k[8], int c, int W, size_t H,
                                              int w0, int w1) {
  uint32_t carry = 0;
  const uint32_t half = 1u << (c - 1);
  for (int w = 0; w < w1 && w < W; w++) {
    uint32_t d = get_bits(k, w * c, c) + carry;
    const bool ng = d > half;
    carry = ng ? 1u : 0u;
    const uint32_t mag = ng ? (1u << c) - d : d;
    if (w < w0 || mag == 0) continue;
    Aff<F> e = T[(size_t)w * H + (mag - 1)];
    if (ng) F::neg(e.y, e.y);
    Jac<F>::add_mixed(acc, acc, e);
  }
}

// (3 resident blocks per SM on G1, 2 on G2: the register budgets the kernel had before the by-value product ABI let the
// callers keep more in registers -- unbounded, G1 grew to 176 registers = 2 blocks and lost 5 %)
template <class F>
__global__ void __launch_bounds__(GS_TAB_NT, sizeof(typename F::T) == sizeof(fp) ? 3 : GS_FC_G2_BLOCKS) k_fixed_commit(const Aff<F>* __restrict__ tab, int c, int W, size_t H, int base0,
                                                            int base1, const fr* __restrict__ s0, size_t s0_stride,
                                                            const fr* __restrict__ s1, size_t s1_stride,
                                                            const Aff<F>* __restrict__ addend, Aff<F>* __restrict__ out, size_t n) {
  __shared__ fp sm[2 * GS_TAB_NT];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = id < 2 * n;
  size_t i = active ? id >> 1 : 0;
  int a = (int)(id & 1);
  Jac<F> acc;
  acc.set_inf();
  if (active) {
    uint32_t k[8];
    fr_from_mont(k, s0[i * s0_stride]);
    fixed_base_accumulate<F>(acc, tab + ((size_t)(base0 * 2 + a) * W) * H, k, c, W, H);
    fr_from_mont(k, s1[i * s1_stride]);
    fixed_base_accumulate<F>(acc, tab + ((size_t)(base1 * 2 + a) * W) * H, k, c, W, H);
    if (addend != nullptr && a == 1) Jac<F>::add_mixed(acc, acc, addend[i]);
  }
  Aff<F> r;
  block_to_affine<GS_TAB_NT>(r, acc, sm);
  if (active) out[i * 2 + a] = r;
}

// ------------------------------------------------------------------ variable-base MSM (proof elements)
// terms[row][t] = sv[row][t] * base[t]   (4-bit signed windows per term), bases = two concatenated segments
// blockIdx.y = proof instance (b1_bs = instance stride of the variable segment, 0 when shared).
// Every term is split along the group's endomorphism (endo.cuh): thread (term, j) multiplies the j-th sub-scalar
// (128 bits on G1, 64 bits on G2) into its own image of the base, so the serial chain of one thread is 32 / 16
// windows instead of 64 and a lone prove is 2 - 4 times shorter; terms[row][t * PARTS + j], summed by reduce_rows.
template <class F>
__global__ void __launch_bounds__(128) k_msm_terms(Jac<F>* __restrict__ terms, const fr* __restrict__ sv, const Aff<F>* __restrict__ b0,
                                                   size_t n0, const Aff<F>* __restrict__ b1, size_t n1, int rows, size_t b1_bs,
                                                   int PARTS /* EndoSplit<F>::PARTS, or 1 = whole scalar per thread */,
                                                   size_t nt /* terms per row in `terms` / `sv`: n0 + n1, or more when the
                                                                variable segment is filled from shared-base tables */) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t nc = n0 + n1;  // terms this launch computes per row
  if (id >= nc * rows * PARTS) return;
  const int j = (int)(id % PARTS);
  const size_t tr = id / PARTS;
  const size_t t = tr % nc, row = tr / nc;
  const size_t term = row * nt + t;
  terms += (size_t)blockIdx.y * nt * rows * PARTS;
  sv += (size_t)blockIdx.y * nt * rows;
  b0 += (size_t)blockIdx.y * n0;
  b1 += (size_t)blockIdx.y * b1_bs;
  Aff<F> B = t < n0 ? b0[t] : b1[t - n0];
  uint32_t k[8];
  fr_from_mont(k, sv[term]);
  Jac<F> r;
  if (PARTS == 1)
    scalar_mul<F>(r, B, k);
  else
    EndoSplit<F>::part(r, B, k, j);
  terms[term * PARTS + j] = r;
}

// ------------------------------------------------------------------ shared-variable window tables (many equations, one witness set)
// A multi-equation statement proves every equation over the SAME variables (C4): sum_j RG[i][j] iota(Y_j) has shared
// bases and per-equation scalars, so the nvars bases get signed 8-bit window tables once per batch
//     T[(j*W + w)*H + d-1] = d * 2^(8w) * V_j      (H = 128; W: below)
// and a variable term costs 32 mixed additions instead of a 255-bit double-and-add.
// The scalars are split along the group's endomorphism (endo.cuh: k = k1 + k2 x^2 on G1, k = sum_j c_j |x|^j on G2), so the
// tables only span the sub-scalars: 128 bits on G1 (16 windows + one for the carry of the signed recoding), 64 bits on G2
// (8 + 1).  The doubling chain that builds the window bases -- one thread per variable, pure latency -- is 128 / 64
// doublings instead of 248 (G2, 64 variables: 7 ms -> 2), the table is 2 / 4 times smaller, and a term costs the same
// number of additions: the sub-scalars are summed Horner-fashion IN the endomorphism,
//     k V = c_0 V + E( c_1 V + E( c_2 V + E( c_3 V ) ) ),   E = -psi on G2 (E = -phi with two sub-scalars on G1),
// E applied to the running Jacobian sum (two / three field products).
constexpr int GS_PT_C = 8, GS_PT_H = 128, GS_PT_RUN = 32;
template <class F>
GS_HD constexpr int ptab_windows() {
  return sizeof(typename F::T) == sizeof(fp) ? 17 : 9;
}
template <class F>
struct PipSplit;  // pippenger.cuh (included below): the sub-scalars of a scalar
// E(P) for a Jacobian point: G1 -phi(X : Y : Z) = (beta X : -Y : Z); G2 -psi(X : Y : Z) = (conj(X) cx : -conj(Y) cy : conj(Z))
GS_HD GS_INL void endo_neg_jac(g1_jac& p) {
  endo_phi_x(p.X, p.X);
  fp::neg(p.Y, p.Y);
}
GS_HD GS_INL void endo_neg_jac(g2_jac& p) {
  g2_aff a, b;
  a.x = p.X;
  a.y = p.Y;
  if (a.is_inf()) fp_one(a.x.c0);  // (endo_psi passes the affine identity (0, 0) through; X = Y = 0 is not a Jacobian point anyway)
  endo_psi(b, a);
  p.X = b.x;
  fp2::neg(p.Y, b.y);
  fp2::conj(p.Z, p.Z);
}
template <class F>
__global__ void __launch_bounds__(128) k_ptab_bases(const Aff<F>* __restrict__ bases, Jac<F>* __restrict__ J, int nb) {
  constexpr int W = ptab_windows<F>();
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  Jac<F> j;
  j.from_affine(bases[b]);
  for (int w = 0; w < W; w++) {
    J[(size_t)b * W + w] = j;
    if (w + 1 < W)
      for (int i = 0; i < GS_PT_C; i++) Jac<F>::dbl(j, j);
  }
}
// thread -> (row (j, w), run r): multiples r*RUN + 1 .. r*RUN + RUN of the row's base tab[row*H]
template <class F>
__global__ void __launch_bounds__(128) k_ptab_fill(const Aff<F>* __restrict__ tab, Jac<F>* __restrict__ J, size_t nrows) {
  constexpr int RUNS = GS_PT_H / GS_PT_RUN;
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nrows * RUNS) return;
  size_t row = id / RUNS;
  int r = (int)(id % RUNS);
  Aff<F> B = tab[row * GS_PT_H];
  Jac<F> acc;
  acc.from_affine(B);
  if (r > 0) {
    Jac<F> step = acc;
    for (int i = 0; i < 5; i++) Jac<F>::dbl(step, step);  // RUN * B
    for (int i = 0; i < r; i++) Jac<F>::add(acc, acc, step);
  }
  Jac<F>* o = J + row * GS_PT_H + (size_t)r * GS_PT_RUN;
  o[0] = acc;
  for (int d = 1; d < GS_PT_RUN; d++) {
    Jac<F>::add_mixed(acc, acc, B);
    o[d] = acc;
  }
}
// thread -> entry: out[idx * ostride] = affine(in[idx]), one field inversion per block
template <class F>
__global__ void __launch_bounds__(128) k_ptab_to_affine(const Jac<F>* __restrict__ in, Aff<F>* __restrict__ out, size_t n, size_t ostride) {
  __shared__ fp sm[2 * 128];
  size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  Jac<F> j;
  j.set_inf();
  if (idx < n) j = in[idx];
  Aff<F> a;
  block_to_affine<128>(a, j, sm);
  if (idx < n) out[idx * ostride] = a;
}
// thread -> (row, variable t) of proof blockIdx.y: terms[row][n0 + t] = sv[row][n0 + t] * V_t from the tables
template <class F>
__global__ void __launch_bounds__(128) k_msm_var_terms_tab(Jac<F>* __restrict__ terms, const fr* __restrict__ sv,
                                                           const Aff<F>* __restrict__ tab, size_t n0, size_t n1, int rows) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= n1 * rows) return;
  const size_t nt = n0 + n1;
  const size_t t = id % n1, row = id / n1;
  const size_t at = (size_t)blockIdx.y * nt * rows + row * nt + n0 + t;
  constexpr int W = ptab_windows<F>(), PARTS = PipSplit<F>::PARTS;
  uint32_t k[8], sub[PARTS][4];
  fr_from_mont(k, sv[at]);
  PipSplit<F>::split(sub, k);
  Jac<F> acc;
  acc.set_inf();
  for (int j = PARTS - 1; j >= 0; j--) {
    if (j != PARTS - 1 && !acc.is_inf()) endo_neg_jac(acc);
    uint32_t kk[8] = {sub[j][0], sub[j][1], sub[j][2], sub[j][3], 0, 0, 0, 0};
    fixed_base_accumulate<F>(acc, tab + (t * W) * GS_PT_H, kk, GS_PT_C, W, (size_t)GS_PT_H);
  }
  terms[at] = acc;
}

// in-place pairwise tree reduction: terms[row][t] += terms[row][t + half] for t < half (one launch per level)
template <class F>
__global__ void __launch_bounds__(128) k_jac_reduce_step(Jac<F>* __restrict__ terms, size_t row_stride, size_t cur, size_t half, int rows) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= half * rows) return;
  terms += (size_t)blockIdx.y * row_stride * rows;
  size_t row = id / half, t = id % half;
  if (t + half >= cur) return;
  Jac<F>* base = terms + row * row_stride;
  Jac<F> a = base[t], b = base[t + half];
  Jac<F>::add(a, a, b);
  base[t] = a;
}

// final assembly of a proof element (prove.rs:146, 162):
//   out[i].p[0] =                  sum_l coef[i][l] key_l.0  (+ e_i W.0)
//   out[i].p[1] = varsum[i]      + sum_l coef[i][l] key_l.1  (+ e_i W.1)
// `varsum` = reduced MSM rows (group-typed) or null; `e` = collapsed scalar (scalar-typed) or null.
// key_l (u_l / v_l) and W are the CRS points the fixed-base window tables hold (bases l and 2): one table
// lookup + mixed addition per window instead of a 255-step double-and-add.
// The CRS-key terms are spread over threads (a lone proof is latency: 64 - 96 dependent additions in
// one thread were 3.2 ms per group): thread -> (i, a, scalar s, window chunk ch) adds PF_WCH windows of ONE scalar,
//   kt[((i*2 + a) * KT) + s*PF_NCH + ch],   KT = nscal * PF_NCH,   scalar s < ncoef: coef[i][s] on key s; s == ncoef: e_i on W
// the partial sums are tree-reduced (reduce_rows) and k_proof_finish2 adds the variable MSM and normalises.
constexpr int PF_NCH = 8;
template <class F>
__global__ void __launch_bounds__(128) k_proof_key_terms(Jac<F>* __restrict__ kt, int rows, int ncoef, const fr* __restrict__ coef,
                                                         const Aff<F>* __restrict__ tab, int c, int W, size_t H, const fr* __restrict__ e,
                                                         int nscal) {
  const int KT = nscal * PF_NCH;
  int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= rows * 2 * KT) return;
  const int ch = id % PF_NCH, sidx = (id / PF_NCH) % nscal, ia = id / KT;
  const int i = ia >> 1, a = ia & 1;
  kt += (size_t)blockIdx.y * rows * 2 * KT;
  coef += (size_t)blockIdx.y * rows * ncoef;
  if (e != nullptr) e += (size_t)blockIdx.y * rows;
  const int wch = (W + PF_NCH - 1) / PF_NCH;
  uint32_t k[8];
  fr_from_mont(k, sidx < ncoef ? coef[i * ncoef + sidx] : e[i]);
  const int base = sidx < ncoef ? sidx : 2;  // table bases: key_0, key_1, W
  Jac<F> acc;
  acc.set_inf();
  fixed_base_accumulate_range<F>(acc, tab + ((size_t)(base * 2 + a) * W) * H, k, c, W, H, ch * wch, (ch + 1) * wch);
  kt[id] = acc;
}
template <class F>
__global__ void k_proof_finish2(Aff<F>* __restrict__ out, int rows, const Jac<F>* __restrict__ kt, int KT, const Jac<F>* __restrict__ varsum,
                                size_t var_stride) {
  int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= rows * 2) return;
  int i = id >> 1, a = id & 1;
  out += (size_t)blockIdx.y * rows * 2;
  kt += (size_t)blockIdx.y * rows * 2 * KT;
  Jac<F> acc = kt[(size_t)id * KT];
  if (varsum != nullptr && a == 1) {
    Jac<F> vs = varsum[(size_t)blockIdx.y * var_stride * rows + (size_t)i * var_stride];
    Jac<F>::add(acc, acc, vs);
  }
  Aff<F> r;
  Jac<F>::to_affine(r, acc);
  out[id] = r;
}

// ------------------------------------------------------------------ rerandomisation of a committed proof
// c' = c + R' u_x (and d' = d + S' v_y): out[i].p[a] = com[i].p[a] + sum_{k < ns} s[i][k] key_k.a from the fixed-base tables.
// Unlike k_fixed_commit the addend is a whole commitment (both coordinates); k_fixed_commit keeps its C2 register budget.
template <class F>
__global__ void __launch_bounds__(GS_TAB_NT) k_rerand_commit(const Aff<F>* __restrict__ tab, int c, int W, size_t H, const fr* __restrict__ s,
                                                             int ns, const Aff<F>* __restrict__ com, Aff<F>* __restrict__ out, size_t n) {
  __shared__ fp sm[2 * GS_TAB_NT];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = id < 2 * n;
  size_t i = active ? id >> 1 : 0;
  int a = (int)(id & 1);
  Jac<F> acc;
  acc.set_inf();
  if (active) {
    acc.from_affine(com[i * 2 + a]);
    for (int k = 0; k < ns; k++) {
      uint32_t kk[8];
      fr_from_mont(kk, s[i * ns + k]);
      fixed_base_accumulate<F>(acc, tab + ((size_t)(k * 2 + a) * W) * H, kk, c, W, H);
    }
  }
  Aff<F> r;
  block_to_affine<GS_TAB_NT>(r, acc, sm);
  if (active) out[i * 2 + a] = r;
}

// out[i].p[a] = com[i].p[a] + s0_i Base0.a + s1_i Base1.a: a whole commitment plus two fixed-base products, the sibling of
// k_fixed_commit (which adds iota(X) to coordinate 1 only and keeps its C2 register budget).  The linear equations
// Z_k - delta P_k = O of a rerandomised zk PPE proof (zk.cu) are pi'_c = pi_c + R'_c W2 - T'_c v1 and
// theta' = theta + T'_0 u1 + T'_1 u2: fixed-base terms only.
template <class F>
__global__ void __launch_bounds__(GS_TAB_NT) k_fixed_com_add(const Aff<F>* __restrict__ tab, int c, int W, size_t H, int base0,
                                                             int base1, const fr* __restrict__ s0, size_t s0_stride,
                                                             const fr* __restrict__ s1, size_t s1_stride,
                                                             const Aff<F>* __restrict__ com, Aff<F>* __restrict__ out, size_t n) {
  __shared__ fp sm[2 * GS_TAB_NT];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = id < 2 * n;
  size_t i = active ? id >> 1 : 0;
  int a = (int)(id & 1);
  Jac<F> acc;
  acc.set_inf();
  if (active) {
    acc.from_affine(com[i * 2 + a]);
    uint32_t k[8];
    fr_from_mont(k, s0[i * s0_stride]);
    fixed_base_accumulate<F>(acc, tab + ((size_t)(base0 * 2 + a) * W) * H, k, c, W, H);
    fr_from_mont(k, s1[i * s1_stride]);
    fixed_base_accumulate<F>(acc, tab + ((size_t)(base1 * 2 + a) * W) * H, k, c, W, H);
  }
  Aff<F> r;
  block_to_affine<GS_TAB_NT>(r, acc, sm);
  if (active) out[i * 2 + a] = r;
}

// Variable-base products of a rerandomised proof element (pi': G2 over the constants B and the commitments d; theta': G1
// over A and c).  Output row i has two coordinate rows:
//   a = 1:  sum_{k < n0} sv[i][k] B_k + sum_j sv[i][c0 + j] com_j.1        (n0 = 0 on a scalar-typed side)
//   a = 0:                              sum_j sv[i][c0 + j] com_j.0
// terms[((y*rows + i)*2 + a)*ns*PARTS + slot*PARTS + part], ns = n0 + ncom slots (slot k < n0: B_k; n0 + j: com_j).
// Only the n0 + 2 ncom real products of a row are computed, product q of [q0, q1):  q < n0: B_q (a = 1);
// q < n0 + ncom: com_{q-n0}.1; else com_{q-n0-ncom}.0.  The n0 constant slots of an a = 0 row are zeroed by the caller.
template <class F>
__global__ void __launch_bounds__(128) k_rerand_terms(Jac<F>* __restrict__ terms, const fr* __restrict__ sv, size_t svs, size_t c0,
                                                      const Aff<F>* __restrict__ b0, size_t n0, const Aff<F>* __restrict__ com, size_t ncom,
                                                      size_t com_bs, int rows, size_t q0, size_t q1, int PARTS) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t nq = q1 - q0;
  if (id >= nq * rows * PARTS) return;
  const int j = (int)(id % PARTS);
  const size_t qr = id / PARTS;
  const size_t q = q0 + qr % nq, i = qr / nq;
  const size_t ntp = (n0 + ncom) * PARTS;
  terms += (size_t)blockIdx.y * rows * 2 * ntp;
  sv += (size_t)blockIdx.y * rows * svs;
  b0 += (size_t)blockIdx.y * n0;
  com += (size_t)blockIdx.y * com_bs;
  Aff<F> B;
  size_t col, slot;
  int a = 1;
  if (q < n0) {
    B = b0[q];
    col = q;
    slot = q;
  } else {
    const size_t t = q - n0;
    const size_t jc = t < ncom ? t : t - ncom;
    a = t < ncom ? 1 : 0;
    B = com[jc * 2 + a];
    col = c0 + jc;
    slot = n0 + jc;
  }
  uint32_t k[8];
  fr_from_mont(k, sv[i * svs + col]);
  Jac<F> r;
  if (PARTS == 1)
    scalar_mul<F>(r, B, k);
  else
    EndoSplit<F>::part(r, B, k, j);
  terms[(i * 2 + a) * ntp + slot * PARTS + j] = r;
}

// Shared commitments (one set for every equation): thread -> (i, a, j) of equation blockIdx.y,
// terms[((y*rows + i)*2 + a)*ns + n0 + j] = sv[i][c0 + j] * com_j.a from the shared-base tables (table row 2j + a).
template <class F>
__global__ void __launch_bounds__(128) k_rerand_com_terms_tab(Jac<F>* __restrict__ terms, const fr* __restrict__ sv, size_t svs, size_t c0,
                                                              const Aff<F>* __restrict__ tab, size_t n0, size_t ncom, int rows) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (size_t)rows * 2 * ncom) return;
  const size_t jc = id % ncom, ia = id / ncom;
  const size_t i = ia >> 1;
  const int a = (int)(ia & 1);
  const size_t ns = n0 + ncom;
  constexpr int W = ptab_windows<F>(), PARTS = PipSplit<F>::PARTS;
  uint32_t k[8], sub[PARTS][4];
  fr_from_mont(k, sv[(size_t)blockIdx.y * rows * svs + i * svs + c0 + jc]);
  PipSplit<F>::split(sub, k);
  Jac<F> acc;
  acc.set_inf();
  for (int p = PARTS - 1; p >= 0; p--) {
    if (p != PARTS - 1 && !acc.is_inf()) endo_neg_jac(acc);
    uint32_t kk[8] = {sub[p][0], sub[p][1], sub[p][2], sub[p][3], 0, 0, 0, 0};
    fixed_base_accumulate<F>(acc, tab + ((jc * 2 + a) * W) * GS_PT_H, kk, GS_PT_C, W, (size_t)GS_PT_H);
  }
  terms[(((size_t)blockIdx.y * rows + i) * 2 + a) * ns + n0 + jc] = acc;
}

// where the variable-base sum of coordinate a of output row i of proof y is: p[a][y * inst[a] + i * row[a]] (p[a] null: none)
template <class F>
struct rerand_sums {
  const Jac<F>* p[2];
  size_t inst[2], row[2];
};
// out[i].p[a] = old[i].p[a] + the key / W terms (reduced kt, as for k_proof_finish2) + the variable-base sum of coordinate a
template <class F>
__global__ void k_rerand_finish(Aff<F>* __restrict__ out, int rows, const Jac<F>* __restrict__ kt, int KT, const Aff<F>* __restrict__ old,
                                rerand_sums<F> vs) {
  int id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= rows * 2) return;
  int i = id >> 1, a = id & 1;
  const size_t y = blockIdx.y;
  out += y * rows * 2;
  old += y * rows * 2;
  kt += y * rows * 2 * KT;
  Jac<F> acc = kt[(size_t)id * KT];
  Jac<F>::add_mixed(acc, acc, old[id]);
  if (vs.p[a] != nullptr) {
    Jac<F> v = vs.p[a][y * vs.inst[a] + (size_t)i * vs.row[a]];
    Jac<F>::add(acc, acc, v);
  }
  Aff<F> r;
  Jac<F>::to_affine(r, acc);
  out[id] = r;
}

// ------------------------------------------------------------------ Mat::left_mul on Com matrices
// terms[(i*c + j)*2 + a][t] = lhs[i][t] * mat[t][j].a      (data_structures.rs:696-742)
template <class F>
__global__ void __launch_bounds__(128) k_com_matmul_terms(Jac<F>* __restrict__ terms, const fr* __restrict__ lhs,
                                                          const Aff<F>* __restrict__ mat, size_t r, size_t k, size_t c) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= r * c * 2 * k) return;
  size_t t = id % k;
  size_t o = id / k;
  int a = (int)(o & 1);
  size_t ij = o >> 1;
  size_t i = ij / c, j = ij % c;
  uint32_t kk[8];
  fr_from_mont(kk, lhs[i * k + t]);
  Jac<F> acc;
  scalar_mul<F>(acc, mat[(t * c + j) * 2 + a], kk);
  terms[id] = acc;
}
template <class F>
__global__ void k_jac_rows_to_affine(Aff<F>* __restrict__ out, const Jac<F>* __restrict__ terms, size_t row_stride, size_t rows) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= rows) return;
  Aff<F> r;
  Jac<F>::to_affine(r, terms[id * row_stride]);
  out[id] = r;
}

}  // namespace gs

namespace gsi {

template <class F>
struct crs_side;
template <>
struct crs_side<FpOps> {
  static const g1_aff* key(const crs_dev* c) { return &c->u[0][0]; }
  static const g1_aff* w(const crs_dev* c) { return &c->w1[0]; }
};
template <>
struct crs_side<Fp2Ops> {
  static const g2_aff* key(const crs_dev* c) { return &c->v[0][0]; }
  static const g2_aff* w(const crs_dev* c) { return &c->w2[0]; }
};

template <class F>
void fixed_table_release(gs_ctx* ctx) {
  gs_fixed_table<F>& T = table_of<F>(ctx);
  if (T.t) cudaFree(T.t);
  T.t = nullptr;
  T.c = 0;
}

// T[w][d-1] = d * 2^(c w) * B for the six base coordinates (u1 u2 W1 / v1 v2 W2); c = 8 at CRS load
// (L2-resident), c = 16 lazily for big batches.
template <class F>
int fixed_table_rebuild(gs_ctx* ctx, int c) {
  gs_fixed_table<F>& T = table_of<F>(ctx);
  fixed_table_release<F>(ctx);
  T.c = c;
  T.W = (256 + c - 1) / c;
  T.H = (size_t)1 << (c - 1);
  size_t n = (size_t)6 * T.W * T.H;
  CUDA_TRY(cudaMalloc(&T.t, n * sizeof(Aff<F>)));
  // the six base points: u[2][2] then w1[2]  (v[2][2] then w2[2])
  Scratch sc(ctx);
  Aff<F>* b;
  CUDA_TRY(sc.alloc(&b, 6));
  const Aff<F>* key = crs_side<F>::key(ctx->crs);
  const Aff<F>* W = crs_side<F>::w(ctx->crs);
  CUDA_TRY(cudaMemcpyAsync(b, key, 4 * sizeof(Aff<F>), cudaMemcpyDeviceToDevice, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(b + 4, W, 2 * sizeof(Aff<F>), cudaMemcpyDeviceToDevice, ctx->stream));
  LAUNCH_CFG((k_table_window_bases<F>), 6, 32, 0, b, T.t, T.c, T.W, T.H);
  constexpr int RUN = 16;
  size_t threads = (size_t)6 * T.W * ((T.H + RUN - 1) / RUN);
  LAUNCH_CFG((k_table_fill<F, RUN>), threads, GS_TAB_NT, 0, T.t, T.W, T.H);
  return GS_OK;
}

// the fixed-base tables for a batch of n commitments: big batches amortise bigger windows, 16 windows of 16 bits instead
// of 32 of 8 (never downgraded: once the c = 16 tables exist, small batches use them too instead of rebuilding c = 8)
template <class F>
int fixed_table_for(gs_ctx* ctx, size_t n) {
  gs_fixed_table<F>& T = table_of<F>(ctx);
  int want_c = n >= 8192 ? 16 : 8;
  if (!T.t || (want_c == 16 && T.c != 16)) return fixed_table_rebuild<F>(ctx, want_c);
  return GS_OK;
}

// out[i] = s0[i] Base0 + s1[i] Base1 (+ iota(addend[i]))    -- all four batch_commit_* variants
template <class F>
int batch_commit_impl(gs_ctx* ctx, size_t n, int base0, int base1, const gs_fr* s0, size_t s0_stride, const gs_fr* s1,
                      size_t s1_stride, size_t nscal, const void* addend, void* out) {
  if (!ctx || !s0 || !out) return GS_EARG;
  if (!ctx->crs_loaded) FAIL(GS_EARG, "commit: no CRS loaded");
  if (n == 0) return GS_OK;  // reference: empty input -> empty Commit (left_mul returns vec![])
  CUDA_TRY(cudaSetDevice(ctx->device));
  int rct = fixed_table_for<F>(ctx, n);
  if (rct) return rct;
  gs_fixed_table<F>& T = table_of<F>(ctx);
  // Big batches (C2: 2^20 variables = 160 MB in, 192 MB out for G1) are cut into chunks that alternate between two
  // streams: while the host stages chunk i+1 in and chunk i-1 out (pageable copies block the host, not the GPU),
  // the kernel of chunk i runs.  Only the interleaved-randomness layout (batch_commit_G1/G2) is chunked.
  const size_t CH = (size_t)1 << 16;
  if (n > 2 * CH && s0_stride == 2 && (const fr*)s1 == (const fr*)s0 + 1 && nscal == 2 * n && addend) {
    if (!ctx->stream2) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
    cudaStream_t main_stream = ctx->stream;
    CUDA_TRY(cudaStreamSynchronize(main_stream));  // table build (if any) is done before the second stream reads it
    struct pending_t {
      Scratch* sc = nullptr;
      Aff<F>* dout = nullptr;
      size_t off = 0, cnt = 0;
      cudaStream_t st = nullptr;
    } prev;
    int rc = GS_OK;
    cudaError_t ce = cudaSuccess;
    auto drain = [&](pending_t& pd) {  // D2H of a finished chunk (blocks until its kernel is done), then release
      if (!pd.sc) return;
      ctx->stream = pd.st;
      cudaError_t e2 = cudaMemcpyAsync((Aff<F>*)out + 2 * pd.off, pd.dout, 2 * pd.cnt * sizeof(Aff<F>), cudaMemcpyDeviceToHost, pd.st);
      if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(pd.st);
      if (ce == cudaSuccess) ce = e2;
      delete pd.sc;
      pd.sc = nullptr;
    };
    size_t idx = 0;
    for (size_t off = 0; off < n && rc == GS_OK && ce == cudaSuccess; off += CH, idx++) {
      const size_t cnt = n - off < CH ? n - off : CH;
      pending_t cur;
      cur.st = (idx & 1) ? ctx->stream2 : main_stream;
      cur.off = off;
      cur.cnt = cnt;
      ctx->stream = cur.st;
      cur.sc = new Scratch(ctx);
      fr* ds;
      Aff<F>* dadd;
      cudaError_t e2 = upload(ctx, *cur.sc, &ds, (const fr*)s0 + 2 * off, 2 * cnt);
      if (e2 == cudaSuccess) e2 = upload(ctx, *cur.sc, &dadd, (const Aff<F>*)addend + off, cnt);
      if (e2 == cudaSuccess) e2 = cur.sc->alloc(&cur.dout, 2 * cnt);
      if (e2 != cudaSuccess) {
        ce = e2;
        delete cur.sc;
        break;
      }
      rc = [&]() -> int {
        LAUNCH((k_fixed_commit<F>), 2 * cnt, T.t, T.c, T.W, T.H, base0, base1, (const fr*)ds, (size_t)2, (const fr*)ds + 1, (size_t)2,
               dadd, cur.dout, cnt);
        return GS_OK;
      }();
      drain(prev);  // overlaps with the kernel just launched on the other stream
      prev = cur;
    }
    drain(prev);
    ctx->stream = main_stream;
    if (rc) return rc;
    CUDA_TRY(ce);
    return GS_OK;
  }
  Scratch sc(ctx);
  fr* ds;
  Aff<F>* dadd = nullptr;
  Aff<F>* dout;
  CUDA_TRY(upload(ctx, sc, &ds, s0, nscal));
  if (addend) CUDA_TRY(upload(ctx, sc, &dadd, addend, n));
  CUDA_TRY(sc.alloc(&dout, 2 * n));
  const fr* d0 = ds;
  const fr* d1 = ds + ((const fr*)s1 - (const fr*)s0);
  LAUNCH((k_fixed_commit<F>), 2 * n, T.t, T.c, T.W, T.H, base0, base1, d0, s0_stride,
         d1, s1_stride, dadd, dout, n);
  CUDA_TRY(cudaMemcpyAsync(out, dout, 2 * n * sizeof(Aff<F>), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

// reduce rows of Jacobian terms in place (row i occupies terms[i*stride .. i*stride+cnt))
template <class F>
int reduce_rows(gs_ctx* ctx, Jac<F>* terms, size_t stride, size_t cnt, int rows, size_t nbatch = 1) {
  size_t cur = cnt;
  while (cur > 1) {
    size_t half = (cur + 1) / 2;
    LAUNCH_B((k_jac_reduce_step<F>), half * rows, nbatch, terms, stride, cur, half, rows);
    cur = half;
  }
  return GS_OK;
}

// the CRS-key terms of the proof elements of `count` proofs (k_proof_key_terms -> tree): the sum of (i, a) lands in
// (*kt)[(i*2 + a) * *KT] of each proof
template <class F>
int proof_key_sums(gs_ctx* ctx, Scratch& sc, size_t count, int rows, int ncoef, const fr* coef, const gs_fixed_table<F>& T,
                   const fr* e, Jac<F>** kt, int* KT) {
  const int nscal = ncoef + (e != nullptr ? 1 : 0);
  *KT = nscal * PF_NCH;
  CUDA_TRY(sc.alloc(kt, count * (size_t)rows * 2 * *KT));
  LAUNCH_B((k_proof_key_terms<F>), (size_t)rows * 2 * *KT, count, *kt, rows, ncoef, coef, T.t, T.c, T.W, T.H, e, nscal);
  return reduce_rows<F>(ctx, *kt, (size_t)*KT, (size_t)*KT, rows * 2, count);
}

// final assembly of the proof elements of `count` proofs (key sums -> k_proof_finish2)
template <class F>
int proof_finish(gs_ctx* ctx, Scratch& sc, size_t count, int rows, int ncoef, const fr* coef, const gs_fixed_table<F>& T,
                 const Jac<F>* varsum, size_t var_stride, const fr* e, Aff<F>* dout) {
  Jac<F>* kt;
  int KT;
  int rc = proof_key_sums<F>(ctx, sc, count, rows, ncoef, coef, T, e, &kt, &KT);
  if (rc) return rc;
  LAUNCH_B((k_proof_finish2<F>), (size_t)rows * 2, count, dout, rows, kt, KT, varsum, var_stride);
  return GS_OK;
}

// shared-base window tables of nb points (see k_ptab_bases): ptab = nb * ptab_windows rows of GS_PT_H affine multiples,
// J = Jacobian scratch of the same size
template <class F>
cudaError_t shared_base_alloc(Scratch& sc, size_t nb, Aff<F>** ptab, Jac<F>** J) {
  const size_t nrows = nb * ptab_windows<F>();
  cudaError_t e = sc.alloc(ptab, nrows * GS_PT_H);
  return e == cudaSuccess ? sc.alloc(J, nrows * GS_PT_H) : e;
}
template <class F>
int shared_base_tables(gs_ctx* ctx, const Aff<F>* bases, size_t nb, Aff<F>* ptab, Jac<F>* J) {
  const size_t nrows = nb * ptab_windows<F>();
  LAUNCH((k_ptab_bases<F>), nb, bases, J, (int)nb);
  LAUNCH((k_ptab_to_affine<F>), nrows, J, ptab, nrows, (size_t)GS_PT_H);
  LAUNCH((k_ptab_fill<F>), nrows * (GS_PT_H / GS_PT_RUN), ptab, J, nrows);
  LAUNCH((k_ptab_to_affine<F>), nrows * GS_PT_H, J, ptab, nrows * GS_PT_H, (size_t)1);
  return GS_OK;
}

}  // namespace gsi
#include "pippenger.cuh"
namespace gsi {

// one proof element vector per proof (pi: F = G2, theta: F = G1), see k_proof_finish; batched over `count` proofs
template <class F>
int proof_element(gs_ctx* ctx, Scratch& sc, size_t count, int rows, bool group_typed, const fr* sv, const void* dconst,
                  size_t nconst, const void* dvars, size_t nvars, bool vars_shared, int ncoef, const fr* coef, size_t coef_rs,
                  const fr* e, Aff<F>* dout) {
  size_t nt = nconst + nvars;
  const gs_fixed_table<F>& T = table_of<F>(ctx);  // built by the first commit / prove under this key (c = 8) or by a big
  if (!T.t) {                                     // commit batch (c = 16)
    int rct = fixed_table_rebuild<F>(ctx, 8);
    if (rct) return rct;
  }
  if (coef_rs != (size_t)ncoef) FAIL(GS_EARG, "prove: coefficient matrix must be dense");
  if (group_typed) {
    // few terms (a lone statement): split every scalar multiplication over PARTS threads to shorten the serial chain;
    // big batches are throughput-bound and keep one thread per term (measured on C4: the split costs ~5 % there)
    // many equations over one witness set: the variable terms come from shared-base window tables (break-even ~20 uses
    // of a base; required here: 64) and every thread takes a whole scalar.  A simulated proof (simulate.cu) has no
    // variable terms (nvars = 0) and takes this branch for the shared scalar vector of its constant terms alone.
    const bool var_tables = vars_shared && count * rows >= 64;
    // ONE big statement: bucket MSM (pippenger.cuh) from ctx->pip_min terms up -- W * N additions per row instead of a
    // windowed scalar multiplication per term
    if (count == 1 && !var_tables && nt >= ctx->pip_min) {
      Jac<F>* rowsum;
      size_t stride;
      int rcp = pippenger_rows<F>(ctx, sc, sv, rows, (const Aff<F>*)dconst, nconst, (const Aff<F>*)dvars, nvars, &rowsum, &stride,
                                  ctx->pip_c);
      if (rcp) return rcp;
      return proof_finish<F>(ctx, sc, count, rows, ncoef, coef, T, rowsum, stride, (const fr*)nullptr, dout);
    }
    const int PARTS = (!var_tables && count * nt * rows < 32768) ? EndoSplit<F>::PARTS : 1;
    const size_t ntp = nt * PARTS;
    Jac<F>* terms;
    CUDA_TRY(sc.alloc(&terms, count * ntp * rows));
    if (!var_tables) {
      LAUNCH_B((k_msm_terms<F>), ntp * rows, count, terms, sv, (const Aff<F>*)dconst, nconst, (const Aff<F>*)dvars, nvars, rows,
               vars_shared ? (size_t)0 : nvars, PARTS, nt);
    } else {
      // the tables are built on the second stream while the constant terms (latency-bound scalar multiplications)
      // run on the main one
      Aff<F>* ptab;
      Jac<F>* J;
      CUDA_TRY(shared_base_alloc<F>(sc, nvars, &ptab, &J));
      SideStream side(ctx);
      if (int rc = side.fork()) return rc;
      if (nvars > 0) {
        int rcb = shared_base_tables<F>(ctx, (const Aff<F>*)dvars, nvars, ptab, J);
        if (rcb) return rcb;
        LAUNCH_B((k_msm_var_terms_tab<F>), nvars * rows, count, terms, sv, ptab, nconst, nvars, rows);
      }
      if (int rc = side.back()) return rc;
      if (nconst * PipSplit<F>::PARTS >= 64 && count >= 16) {
        // shared witnesses = shared commitment randomness: the constants of ALL equations are multiplied by the same
        // scalar vector, so the bucket lists are built once and every equation sums its points along them
        // (pippenger.cuh, "ONE scalar vector").  The sum lands in term slot 0, the other constant slots are identities.
        for (int row = 0; row < rows; row++)
          CUDA_TRY(cudaMemset2DAsync(terms + (size_t)row * nt, nt * rows * sizeof(Jac<F>), 0, nconst * sizeof(Jac<F>), count,
                                     ctx->stream));
        int rcs = shared_scalar_sums<F>(ctx, sc, sv, nt, rows, (const Aff<F>*)dconst, nconst, count, terms, nt);
        if (rcs) return rcs;
      } else {
        LAUNCH_B((k_msm_terms<F>), nconst * rows, count, terms, sv, (const Aff<F>*)dconst, nconst, (const Aff<F>*)dvars, (size_t)0, rows,
                 (size_t)0, 1, nt);
      }
      if (int rc = side.join()) return rc;
    }
    int rc = reduce_rows<F>(ctx, terms, ntp, ntp, rows, count);
    if (rc) return rc;
    return proof_finish<F>(ctx, sc, count, rows, ncoef, coef, T, terms, ntp, (const fr*)nullptr, dout);
  } else {
    // scalar-typed side: the caller collapsed the terms into e_i = <sv_i, (consts | vars)> (k_fr_dot, prover.cu)
    return proof_finish<F>(ctx, sc, count, rows, ncoef, coef, T, (const Jac<F>*)nullptr, (size_t)0, e, dout);
  }
}

// c' = c + R' key for n commitments of one group, R' n x ns (ns = 2: u1 u2 / v1 v2; 1: u1 / v1); device buffers
template <class F>
int rerand_commit(gs_ctx* ctx, size_t n, int ns, const fr* dR, const Aff<F>* dcom, Aff<F>* dout) {
  int rc = fixed_table_for<F>(ctx, n);
  if (rc) return rc;
  const gs_fixed_table<F>& T = table_of<F>(ctx);
  LAUNCH((k_rerand_commit<F>), 2 * n, T.t, T.c, T.W, T.H, dR, ns, dcom, dout, n);
  return GS_OK;
}

// out[i] = com[i] + s0_i Base0 + s1_i Base1 for n commitments (k_fixed_com_add); device buffers
template <class F>
int fixed_com_add(gs_ctx* ctx, size_t n, int base0, int base1, const fr* s0, size_t s0_stride, const fr* s1, size_t s1_stride,
                  const Aff<F>* dcom, Aff<F>* dout) {
  int rc = fixed_table_for<F>(ctx, n);
  if (rc) return rc;
  const gs_fixed_table<F>& T = table_of<F>(ctx);
  LAUNCH((k_fixed_com_add<F>), 2 * n, T.t, T.c, T.W, T.H, base0, base1, s0, s0_stride, s1, s1_stride, dcom, dout, n);
  return GS_OK;
}

// One rerandomised proof element vector per proof (pi': F = G2, theta': F = G1), batched over `count` proofs:
//   out[i] = old[i] + (variable-base sums, see k_rerand_terms) + sum_l coef[i][l] key_l (+ e_i W)
// sv = [count][rows][nconst + ncom]: the scalars of the constants, then those of the commitments; rg = the commitment
// columns alone, [count][rows][ncom]; dcom = [count][ncom] Com, or one set for every proof with coms_shared.
// The paths are proof_element's: bucket MSMs for one big statement, shared-base tables over the 2 ncom commitment
// points when many equations share them, else one (split) scalar multiplication per product.
template <class F>
int rerand_element(gs_ctx* ctx, Scratch& sc, size_t count, int rows, bool group_typed, const fr* sv, const fr* rg,
                   const void* dconst, size_t nconst, const Aff<F>* dcom, size_t ncom, bool coms_shared, int ncoef,
                   const fr* coef, const fr* e, const Aff<F>* dold, Aff<F>* dout) {
  if (!table_of<F>(ctx).t) {
    int rct = fixed_table_rebuild<F>(ctx, 8);
    if (rct) return rct;
  }
  const gs_fixed_table<F>& T = table_of<F>(ctx);
  const Aff<F>* B = (const Aff<F>*)dconst;
  const size_t n0 = group_typed ? nconst : 0, svs = nconst + ncom;
  const size_t nprod = n0 + 2 * ncom, ns = n0 + ncom;  // products and term slots of a coordinate row
  const bool var_tables = coms_shared && count * rows >= 64;
  rerand_sums<F> vs;
  if (count == 1 && !var_tables && ns >= ctx->pip_min) {
    Aff<F>*c0, *c1;
    CUDA_TRY(sc.alloc(&c0, ncom));
    CUDA_TRY(sc.alloc(&c1, ncom));
    const size_t A = sizeof(Aff<F>);
    CUDA_TRY(cudaMemcpy2DAsync(c0, A, dcom, 2 * A, A, ncom, cudaMemcpyDeviceToDevice, ctx->stream));
    CUDA_TRY(cudaMemcpy2DAsync(c1, A, dcom + 1, 2 * A, A, ncom, cudaMemcpyDeviceToDevice, ctx->stream));
    Jac<F>*s0, *s1;
    size_t st0, st1;
    int rc = group_typed ? pippenger_rows<F>(ctx, sc, sv, rows, B, n0, c1, ncom, &s1, &st1, ctx->pip_c)
                         : pippenger_rows<F>(ctx, sc, rg, rows, c1, ncom, (const Aff<F>*)nullptr, 0, &s1, &st1, ctx->pip_c);
    if (rc) return rc;
    rc = pippenger_rows<F>(ctx, sc, rg, rows, c0, ncom, (const Aff<F>*)nullptr, 0, &s0, &st0, ctx->pip_c);
    if (rc) return rc;
    vs = {{s0, s1}, {0, 0}, {st0, st1}};
  } else {
    const int PARTS = (!var_tables && count * nprod * rows < 32768) ? EndoSplit<F>::PARTS : 1;
    const size_t ntp = ns * PARTS;
    Jac<F>* terms;
    CUDA_TRY(sc.alloc(&terms, count * rows * 2 * ntp));
    // shared commitment randomness: the constants of all equations along one bucket structure (as in proof_element),
    // the sum in slot 0 of the a = 1 row
    const bool const_sums = var_tables && n0 * PipSplit<F>::PARTS >= 64 && count >= 16;
    // identities in the constant slots no product writes: those of the a = 0 rows, with const_sums those of every row
    if (n0 > 0)
      CUDA_TRY(cudaMemset2DAsync(terms, (const_sums ? 1 : 2) * ntp * sizeof(Jac<F>), 0, n0 * PARTS * sizeof(Jac<F>),
                                 count * rows * (const_sums ? 2 : 1), ctx->stream));
    if (!var_tables) {
      LAUNCH_B((k_rerand_terms<F>), (size_t)rows * nprod * PARTS, count, terms, sv, svs, nconst, B, n0, dcom, ncom,
               coms_shared ? (size_t)0 : 2 * ncom, rows, (size_t)0, nprod, PARTS);
    } else {
      // the commitment tables are built on the second stream while the constant terms run on the main one
      Aff<F>* ptab;
      Jac<F>* J;
      CUDA_TRY(shared_base_alloc<F>(sc, 2 * ncom, &ptab, &J));
      SideStream side(ctx);
      if (int rc = side.fork()) return rc;
      int rcb = shared_base_tables<F>(ctx, dcom, 2 * ncom, ptab, J);
      if (rcb) return rcb;
      LAUNCH_B((k_rerand_com_terms_tab<F>), (size_t)rows * 2 * ncom, count, terms, sv, svs, nconst, ptab, n0, ncom, rows);
      if (int rc = side.back()) return rc;
      if (n0 > 0 && const_sums) {
        int rcs = shared_scalar_sums<F>(ctx, sc, sv, svs, rows, B, n0, count, terms + ntp, 2 * ntp);
        if (rcs) return rcs;
      } else if (n0 > 0) {
        LAUNCH_B((k_rerand_terms<F>), (size_t)rows * n0, count, terms, sv, svs, nconst, B, n0, dcom, ncom, (size_t)0, rows,
                 (size_t)0, n0, 1);
      }
      if (int rc = side.join()) return rc;
    }
    int rc = reduce_rows<F>(ctx, terms, ntp, ntp, rows * 2, count);
    if (rc) return rc;
    vs.p[0] = terms;
    vs.p[1] = terms + ntp;
    vs.inst[0] = vs.inst[1] = (size_t)rows * 2 * ntp;
    vs.row[0] = vs.row[1] = 2 * ntp;
  }
  Jac<F>* kt;
  int KT;
  int rc = proof_key_sums<F>(ctx, sc, count, rows, ncoef, coef, T, e, &kt, &KT);
  if (rc) return rc;
  LAUNCH_B((k_rerand_finish<F>), (size_t)rows * 2, count, dout, rows, kt, KT, dold, vs);
  return GS_OK;
}

template <class F>
int com_matmul_impl(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* lhs, const void* mat, void* out) {
  if (!ctx || !lhs || !mat || !out) return GS_EARG;
  // reference: empty operands give an empty matrix (data_structures.rs:697-702)
  if (r == 0 || k == 0 || c == 0) return GS_OK;
  if (r * c * k > ((size_t)1 << 26)) FAIL(GS_EDIM, "matmul: too large");
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  fr* dl;
  Aff<F>*dm, *dout;
  Jac<F>* terms;
  CUDA_TRY(upload(ctx, sc, &dl, lhs, r * k));
  CUDA_TRY(upload(ctx, sc, &dm, mat, k * c * 2));
  CUDA_TRY(sc.alloc(&dout, r * c * 2));
  CUDA_TRY(sc.alloc(&terms, r * c * 2 * k));
  LAUNCH((k_com_matmul_terms<F>), r * c * 2 * k, terms, dl, dm, r, k, c);
  int rc = reduce_rows<F>(ctx, terms, k, k, (int)(r * c * 2));
  if (rc) return rc;
  LAUNCH((k_jac_rows_to_affine<F>), r * c * 2, dout, terms, k, r * c * 2);
  CUDA_TRY(cudaMemcpyAsync(out, dout, r * c * 2 * sizeof(Aff<F>), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}


}  // namespace gsi
