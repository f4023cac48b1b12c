// Verifiable::verify for the four equation types (src/verifier.rs:23-157): slot assembly, the G1-side
// statement MSM (re-association of verifier.rs:39-42, SURVEY.md §8a), then the pairing-product pipeline.
#include <algorithm>

#include "batchinv.cuh"
#include "ctx.h"
#include "endo.cuh"
#include "prover_impl.cuh"  // fixed_base_accumulate
#include "randfold.cuh"

using namespace gs;

namespace gs {

// ------------------------------------------------------------------ verify: slot assembly
// thread -> (p, k): fills every slot that is a plain copy / negation.  X slots [0,n), the scalar-B
// slot and the Quad target slot are written later by k_vmsm_reduce.
__global__ void k_verify_assemble(verify_shape s, verify_args v, const crs_dev* __restrict__ crs, g1_aff* __restrict__ X,
                                  g2_aff* __restrict__ Y, size_t nprob) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nprob * (size_t)s.K) return;
  size_t p = id % nprob;
  int k = (int)(id / nprob);
  const int K = s.K;
  g1_aff x0, x1;
  g2_aff y0, y1;
  bool writeX = true;
  if (k < s.n) {  // (P_j, d_j)
    writeX = false;
    y0 = v.ycoms[(p * s.n + k) * 2 + 0];
    y1 = v.ycoms[(p * s.n + k) * 2 + 1];
  } else if (k < s.sPi) {
    if (s.groupB) {  // (c_i, (O, B_i))
      int i = k - s.sB;
      x0 = v.xcoms[(p * s.m + i) * 2 + 0];
      x1 = v.xcoms[(p * s.m + i) * 2 + 1];
      y0.set_inf();
      y1 = ((const g2_aff*)v.b_consts)[p * s.m + i];
    } else {  // (sum_i b_i c_i, W2)
      writeX = false;
      y0 = crs->w2[0];
      y1 = crs->w2[1];
    }
  } else if (k < s.sTh) {  // (-u_k, pi_k)
    int j = k - s.sPi;
    x0 = crs->neg_u[j][0];
    x1 = crs->neg_u[j][1];
    y0 = v.pi[(p * s.cx + j) * 2 + 0];
    y1 = v.pi[(p * s.cx + j) * 2 + 1];
  } else if (k < s.sT) {  // (-theta_k, v_k)
    int j = k - s.sTh;
    x0 = v.theta[(p * s.cy + j) * 2 + 0];
    x1 = v.theta[(p * s.cy + j) * 2 + 1];
    fp::neg(x0.y, x0.y);
    fp::neg(x1.y, x1.y);
    y0 = crs->v[j][0];
    y1 = crs->v[j][1];
  } else {  // target slot
    if (s.type == 1) {  // (-(O, t), W2)
      x0.set_inf();
      x1 = ((const g1_aff*)v.target)[p];
      fp::neg(x1.y, x1.y);
      y0 = crs->w2[0];
      y1 = crs->w2[1];
    } else if (s.type == 2) {  // (-W1, (O, t))
      x0 = crs->neg_w1[0];
      x1 = crs->neg_w1[1];
      y0.set_inf();
      y1 = ((const g2_aff*)v.target)[p];
    } else {  // Quad: (-(t W1), W2)
      writeX = false;
      y0 = crs->w2[0];
      y1 = crs->w2[1];
    }
  }
  if (writeX) {
    X[((size_t)0 * K + k) * nprob + p] = x0;
    X[((size_t)1 * K + k) * nprob + p] = x1;
  }
  Y[((size_t)0 * K + k) * nprob + p] = y0;
  Y[((size_t)1 * K + k) * nprob + p] = y1;
}

// ------------------------------------------------------------------ verify: G1-side statement MSM (v2)
// P_j = iota(A_j) + sum_i Gamma_ij c_i      (re-association of verifier.rs:39-42, SURVEY.md §8a ‡)
// Signed 4-bit windows (Straus: the 4 doublings per window are shared by all bases of the chunk).
// The odd/even multiples 1B..8B of every base are built ONCE per problem by k_vmsm_tables and shared by
// all n outputs; v1's binary double-and-add left half the lanes of every addition idle.
// base index i of problem p, coordinate a:  i < m -> xcoms[p][i].a ;  i == m (scalar A) -> W1.a
__device__ GS_INL g1_aff vmsm_base(const verify_shape& s, const verify_args& v, const crs_dev* crs, size_t p, int i, int a) {
  if (s.na == 1) return v.xfold[p * s.nbases + i];
  if (i < s.m) return v.xcoms[(p * s.m + i) * 2 + a];
  return crs->w1[a];
}
// thread -> (p, i, a): tab[((i*2 + a)*8 + d) * nprob + p] = (d+1) * base
// GLV: k P = k1 P + k2 (-phi(P)) with k = k1 + k2 x^2 (k1, k2 < 2^128), phi(x, y) = (beta x, y) = -[x^2] P on G1
// (the relation serial.cu's membership test uses).  The multiples of -phi(B) share y (negated) with those of B and
// have x' = beta x, stored in tabx by k_vmsm_tables; the Straus loop then runs 32 windows instead of 64.
// biased 128-bit scalar k' = k + 0x88..8 (32 nibbles): digit_w = nibble_w(k') - 8 in [-8, 7] for w < 32, digit_32 = carry
__device__ GS_INL void glv_bias(uint32_t out[5], const uint32_t k[4]) {
  uint32_t carry = 0;
#pragma unroll
  for (int w = 0; w < 4; w++) {
    uint64_t t = (uint64_t)k[w] + 0x88888888u + carry;
    out[w] = (uint32_t)t;
    carry = (uint32_t)(t >> 32);
  }
  out[4] = carry;
}

__global__ void __launch_bounds__(128) k_vmsm_tables(verify_shape s, verify_args v, const crs_dev* __restrict__ crs,
                                                     g1_aff* __restrict__ tab, fp* __restrict__ tabx, size_t nprob) {
  __shared__ fp sm[2 * 128];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int na = s.na;
  bool active = id < nprob * (size_t)s.nb_own() * na;
  size_t p = active ? id % nprob : 0;
  size_t r = active ? id / nprob : 0;
  int a = (int)(r % na), i = (int)(r / na);  // i = index among this rank's bases (table row); base_at(i) = the base
  g1_aff B;
  B.set_inf();
  if (active) B = vmsm_base(s, v, crs, p, s.base_at(i), a);
  // all GS_VTAB multiples in Jacobian form, then ONE batched inversion (Montgomery's trick over the thread's
  // own Z values, block_batch_inv over the per-thread products) instead of one Fermat inversion per multiple
  g1_jac mlt[GS_VTAB];
  mlt[0].from_affine(B);
  g1_jac::dbl(mlt[1], mlt[0]);
  for (int d = 2; d < GS_VTAB; d++) g1_jac::add_mixed(mlt[d], mlt[d - 1], B);
  fp pre[GS_VTAB], z;
  for (int d = 0; d < GS_VTAB; d++) {
    z = mlt[d].Z;
    if (z.is_zero()) fp_one(z);
    if (d == 0)
      pre[0] = z;
    else
      fp::mul(pre[d], pre[d - 1], z);
  }
  fp inv = pre[GS_VTAB - 1];
  block_batch_inv<128>(inv, sm);
  g1_aff* out = tab + ((size_t)(i * na + a) * GS_VTAB) * nprob + p;
  for (int d = GS_VTAB - 1; d >= 0; d--) {
    fp zi;
    if (d > 0)
      fp::mul(zi, inv, pre[d - 1]);
    else
      zi = inv;
    z = mlt[d].Z;
    if (z.is_zero()) fp_one(z);
    fp::mul(inv, inv, z);
    g1_aff e;
    g1_jac::to_affine_with_zinv(e, mlt[d], zi);
    fp bx;
    endo_phi_x(bx, e.x);
    if (active) {
      out[(size_t)d * nprob] = e;
      tabx[((size_t)(i * na + a) * GS_VTAB + d) * nprob + p] = bx;
    }
  }
}

// scalar that multiplies base i in MSM output jj of problem p (false: no such term)
__device__ GS_INL bool vmsm_scalar(fr& sv, const verify_shape& s, const verify_args& v, size_t p, int i, int jj) {
  if (jj < s.n) {  // P_j: Gamma column j, plus a_j on the extra base W1 when A is scalar
    sv = i < s.m ? v.gamma[(p * s.gm + (s.bworld <= 1 ? i : i / s.bworld)) * s.n + jj] : ((const fr*)v.a_consts)[p * s.n + jj];
    return true;
  }
  if (jj == s.n && !s.groupB) {  // C_B = sum_i b_i c_i
    if (i >= s.m) return false;
    sv = ((const fr*)v.b_consts)[p * s.m + i];
    return true;
  }
  if (i != s.m) return false;  // Quad target: t * W1  (W1 is base index m)
  sv = ((const fr*)v.target)[p];
  return true;
}

#ifndef VP_BLOCKS
#define VP_BLOCKS 4
#endif
// thread -> (p, jj, a, chunk)
__global__ void __launch_bounds__(128, VP_BLOCKS) k_vmsm_partial(verify_shape s, verify_args v, const g1_aff* __restrict__ tab,
                                                      const fp* __restrict__ tabx, g1_jac* __restrict__ part, size_t nprob) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_own = s.n_out_owned();  // sharded statement: the other outputs' Miller pairs run on other ranks
  const int na = s.na;
  size_t total = nprob * (size_t)n_own * na * s.nchunk;
  if (id >= total) return;
  size_t p = id % nprob;
  size_t r = id / nprob;
  int a = (int)(r % na);
  r /= na;
  int jj = s.owned_out((int)(r % n_own));
  int ch = (int)(r / n_own);

  // GLV halves of every scalar, biased for the signed 4-bit recoding (glv_bias): entry 2c = k1 (base B), 2c + 1 = k2 (-phi(B))
  uint32_t sc[2 * GS_MSM_CHUNK][5];
  int bidx[GS_MSM_CHUNK];
  int cnt = 0;
  int i0 = ch * s.chunk, i1 = min(s.nb_own(), i0 + s.chunk);
  for (int i = i0; i < i1; i++) {  // i = index among this rank's bases = table row
    fr sv;
    bool have = vmsm_scalar(sv, s, v, p, s.base_at(i), jj);
    if (!have || sv.is_zero()) continue;
    uint32_t k[8], k1[4], k2[4];
    fr_from_mont(k, sv);
    glv_split(k1, k2, k);
    glv_bias(sc[2 * cnt], k1);
    glv_bias(sc[2 * cnt + 1], k2);
    bidx[cnt] = i;
    cnt++;
  }
  g1_jac acc;
  acc.set_inf();
  if (cnt > 0) {
    // The table entry of step (w, i) is fetched one step ahead: its address depends only on the digits, and the
    // load then overlaps the previous (out-of-line) addition instead of stalling in front of its own.
    g1_aff cur, nxt;
    bool cur_nz = false, cur_neg = false, nxt_nz = false, nxt_neg = false;
    auto fetch = [&](int w, int i, g1_aff& e, bool& nz, bool& ng) {
      const int d = (int)((sc[i][w >> 3] >> ((w & 7) * 4)) & 15u) - (w == 32 ? 0 : 8);
      nz = d != 0;
      if (!nz) return;
      const int mag = d < 0 ? -d : d;
      const bool phi = i & 1;
      const size_t at = ((size_t)(bidx[i >> 1] * na + a) * GS_VTAB + (mag - 1)) * nprob + p;
      e.y = tab[at].y;
      e.x = phi ? tabx[at] : tab[at].x;
      ng = (d < 0) != phi;  // the phi half adds multiples of -phi(B) = (beta x, -y)
    };
    fetch(32, 0, cur, cur_nz, cur_neg);
    for (int w = 32; w >= 0; w--) {
      if (w != 32) {
        g1_jac::dbl(acc, acc);
        g1_jac::dbl(acc, acc);
        g1_jac::dbl(acc, acc);
        g1_jac::dbl(acc, acc);
      }
      for (int i = 0; i < 2 * cnt; i++) {
        int ni = i + 1, nw = w;
        if (ni == 2 * cnt) {
          ni = 0;
          nw = w - 1;
        }
        nxt_nz = false;
        if (nw >= 0) fetch(nw, ni, nxt, nxt_nz, nxt_neg);
        if (cur_nz) {
          if (cur_neg) fp::neg(cur.y, cur.y);
          g1_jac::add_mixed(acc, acc, cur);
        }
        cur = nxt;
        cur_nz = nxt_nz;
        cur_neg = nxt_neg;
      }
    }
  }
  part[(((size_t)ch * s.n_out + jj) * na + a) * nprob + p] = acc;
}

// ------------------------------------------------------------------ verify: shared-base window tables
// When ONE set of commitments c_i serves many MSM outputs (a big statement: n outputs per base; or a batch of
// equations over the same commitments, C4), the bases get fixed-base treatment: signed 8-bit window tables
//     T[b][w][d-1] = d * 2^(8w) * base_b,   b = i*2 + a,  w < 32,  d = 1..128      (layout of prover_impl.cuh)
// are built once (4,096 additions per base coordinate) and every scalar product costs 32 mixed additions and no
// doubling, against ~60 additions + a share of 256 doublings in the Straus kernel above.  Break-even is at
// ~160 outputs per base; C3 has 1,024 (2.1 M products: 147 M -> 75 M point additions).
// Window width: c = 8 (32 windows x 128 entries), or c = 10 (26 x 512) when a base serves >= 4,096 outputs -- a batch of
// equations over shared commitments (C4: 16,384 outputs per base) -- where 19 % fewer additions outweigh the 3x table.
struct wt_geom {
  int c, W, H;
};
// The scalars are split along the G1 endomorphism (k = k1 + k2 x^2, k1, k2 < 2^127.4; endo.cuh), so the tables only span
// 128 bits: HALF the windows -- half the doublings, half the table entries to build and to keep -- for the same number of
// additions per scalar (k1's digits select from the table as it is, k2's digits go to a second accumulator that is mapped
// through -phi once per thread at the end).  c = 8: 16 windows + one for the carry of the signed recoding out of the top
// window (its digits are 0 / 1); c = 10: 13 windows cover 130 bits and the top digit is < 2^8, no carry.
static inline wt_geom wt_choose(size_t outputs_per_base) {
  return outputs_per_base >= 4096 ? wt_geom{10, 13, 512} : wt_geom{8, 17, 128};
}
// thread -> flat base b: J[b*W + w] = 2^(8w) * base_b   (one Jacobian doubling chain)
__global__ void __launch_bounds__(128) k_wtab_bases(verify_shape s, verify_args v, const crs_dev* __restrict__ crs,
                                                    g1_jac* __restrict__ J, int nb, wt_geom g) {
  int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= nb) return;
  g1_aff B = vmsm_base(s, v, crs, 0, s.base_at(b / s.na), b % s.na);
  g1_jac j;
  j.from_affine(B);
  for (int w = 0; w < g.W; w++) {
    J[(size_t)b * g.W + w] = j;
    if (w + 1 < g.W)
      for (int i = 0; i < g.c; i++) g1_jac::dbl(j, j);
  }
}
// thread -> (row (b, w), run r): the multiples d = r*RUN + 1 .. r*RUN + RUN of the row's base B = tab[row*H]:
// start (r*RUN + 1) B = B + r * (RUN B) (5 doublings, <= 3 additions), then RUN - 1 mixed additions; 4 runs per row
// keep the dependent chain short (the kernel is latency-bound: 65 k rows are a fraction of one wave).
constexpr int GS_WT_RUN = 32;
__global__ void __launch_bounds__(128) k_wtab_fill(const g1_aff* __restrict__ tab, g1_jac* __restrict__ J, size_t nrows, int H) {
  const int RUNS = H / GS_WT_RUN;
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nrows * RUNS) return;
  size_t row = id / RUNS;
  int r = (int)(id % RUNS);
  g1_aff B = tab[row * H];
  g1_jac acc;
  acc.from_affine(B);
  if (r > 0) {
    g1_jac step = acc;
    for (int i = 0; i < 5; i++) g1_jac::dbl(step, step);  // RUN * B
    for (int i = 0; i < r; i++) g1_jac::add(acc, acc, step);
  }
  g1_jac* o = J + row * H + (size_t)r * GS_WT_RUN;
  o[0] = acc;
  for (int d = 1; d < GS_WT_RUN; d++) {
    g1_jac::add_mixed(acc, acc, B);
    o[d] = acc;
  }
}
// thread -> strip of ST consecutive entries: out[idx * ostride] = affine(in[idx]).  Montgomery's trick inside the
// strip, then across the block (batchinv.cuh): one field inversion per 128 * ST points.
template <int ST>
__global__ void __launch_bounds__(128) k_jac_to_affine_blocks(const g1_jac* __restrict__ in, g1_aff* __restrict__ out, size_t n,
                                                              size_t ostride) {
  __shared__ fp sm[2 * 128];
  const size_t i0 = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * ST;
  fp pre[ST];  // pre[t] = z_0 ... z_t over the strip (infinity / out of range counts as 1)
  fp acc;
  fp_one(acc);
#pragma unroll
  for (int t = 0; t < ST; t++) {
    if (i0 + t < n) {
      fp z = in[i0 + t].Z;
      if (!z.is_zero()) fp::mul(acc, acc, z);
    }
    pre[t] = acc;
  }
  block_batch_inv<128>(acc, sm);  // acc = 1 / (z_0 ... z_{ST-1})
#pragma unroll
  for (int t = ST - 1; t >= 0; t--) {
    if (i0 + t >= n) continue;
    g1_jac j = in[i0 + t];
    g1_aff a;
    if (j.Z.is_zero()) {
      a.set_inf();
    } else {
      fp zi;
      if (t > 0)
        fp::mul(zi, acc, pre[t - 1]);
      else
        zi = acc;
      fp::mul(acc, acc, j.Z);
      g1_jac::to_affine_with_zinv(a, j, zi);
    }
    out[(i0 + t) * ostride] = a;
  }
}
// thread -> (p, jj, a, chunk): same outputs as k_vmsm_partial, bases looked up in the shared tables
__global__ void __launch_bounds__(128, 4) k_vmsm_wsum(verify_shape s, verify_args v, const g1_aff* __restrict__ tab,
                                                   g1_jac* __restrict__ part, size_t nprob, wt_geom g) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int n_own = s.n_out_owned();  // sharded statement: the other outputs' Miller pairs run on other ranks
  const int na = s.na;
  size_t total = nprob * (size_t)n_own * na * s.nchunk;
  if (id >= total) return;
  size_t p = id % nprob;
  size_t r = id / nprob;
  int a = (int)(r % na);
  r /= na;
  int jj = s.owned_out((int)(r % n_own));
  int ch = (int)(r / n_own);
  g1_jac acc, acc2;  // acc: the k1 halves; acc2: the k2 halves, mapped through -phi at the end (phi is additive)
  acc.set_inf();
  acc2.set_inf();
  int i0 = ch * s.chunk, i1 = min(s.nb_own(), i0 + s.chunk);
  for (int i = i0; i < i1; i++) {  // i = index among this rank's bases = table row
    fr sv;
    if (!vmsm_scalar(sv, s, v, p, s.base_at(i), jj) || sv.is_zero()) continue;
    uint32_t k[8], k1[8], k2[8];
    fr_from_mont(k, sv);
    glv_split(k1, k2, k);
#pragma unroll
    for (int t = 4; t < 8; t++) k1[t] = k2[t] = 0;
    const g1_aff* T = tab + ((size_t)(i * na + a) * g.W) * g.H;
    fixed_base_accumulate<FpOps>(acc, T, k1, g.c, g.W, (size_t)g.H);
    fixed_base_accumulate<FpOps>(acc2, T, k2, g.c, g.W, (size_t)g.H);
  }
  if (!acc2.is_inf()) {  // -phi(X : Y : Z) = (beta X : -Y : Z)
    endo_phi_x(acc2.X, acc2.X);
    fp::neg(acc2.Y, acc2.Y);
    g1_jac::add(acc, acc, acc2);
  }
  part[(((size_t)ch * s.n_out + jj) * na + a) * nprob + p] = acc;
}

// thread -> (group g of F chunks, entry e = (jj*2 + a)*nprob + p): out[g][e] = sum_{c < F} part[g*F + c][e]
__global__ void __launch_bounds__(128) k_vmsm_fold(verify_shape s, const g1_jac* __restrict__ part, g1_jac* __restrict__ out,
                                                   size_t nprob, int nchunk, int F, int ngroups) {
  const size_t E = (size_t)s.n_out * s.na * nprob;
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= E * ngroups) return;
  size_t e = id % E;
  int g = (int)(id / E);
  int jj = (int)(e / (s.na * nprob));
  if (!s.owns(s.out_slot(jj))) return;
  int c0 = g * F, c1 = min(nchunk, c0 + F);
  g1_jac acc = part[(size_t)c0 * E + e];
  for (int c = c0 + 1; c < c1; c++) {
    g1_jac t = part[(size_t)c * E + e];
    g1_jac::add(acc, acc, t);
  }
  out[(size_t)g * E + e] = acc;
}

// thread -> (p, jj, a): sum the chunk partials, add iota_1(A_j), negate the Quad target, normalise, write slot
__global__ void __launch_bounds__(128) k_vmsm_reduce(verify_shape s, verify_args v, const g1_jac* __restrict__ part,
                                                     g1_aff* __restrict__ X, size_t nprob) {
  __shared__ fp sm[2 * 128];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int na = s.na;
  bool active = id < nprob * (size_t)s.n_out_owned() * na;
  size_t p = active ? id % nprob : 0;
  size_t r = active ? id / nprob : 0;
  int a = (int)(r % na);
  int jj = active ? s.owned_out((int)(r / na)) : 0;
  g1_jac acc;
  acc.set_inf();
  int slot = 0;
  if (active) {
    acc = part[((size_t)jj * na + a) * nprob + p];
    for (int ch = 1; ch < s.nchunk; ch++) {
      g1_jac t = part[(((size_t)ch * s.n_out + jj) * na + a) * nprob + p];
      g1_jac::add(acc, acc, t);
    }
    if (jj < s.n) {
      slot = jj;
      if (s.groupA && (a == 1 || na == 1)) {  // iota_1(A_j) = (O, A_j); folded: tau_p A_j
        g1_aff A = na == 1 ? v.afold[p * s.n + jj] : ((const g1_aff*)v.a_consts)[p * s.n + jj];
        g1_jac::add_mixed(acc, acc, A);
      }
    } else if (jj == s.n && !s.groupB) {
      slot = s.sB;
    } else {
      slot = s.sT;
      g1_jac::neg(acc, acc);
    }
  }
  g1_aff out;
  block_to_affine<128>(out, acc, sm);
  if (!active) return;
  if (na == 1) {
    const int fm = v.fold_map[slot];
    if (fm >= 0)
      v.fold_X1[p * v.fold_Kw + fm] = out;
    else
      v.fold_Xfix[(size_t)(-fm - 1) * nprob + p] = out;
  } else {
    X[((size_t)a * s.K + slot) * nprob + p] = out;
  }
}

// ---- MSM sharded by base (gs_verify_sharded): the partial sums travel between the ranks as affine points
// thread -> (p, jj, a): parts[(p*n_out + jj)*2 + a] = affine( sum over this rank's chunks )
__global__ void __launch_bounds__(128) k_vmsm_parts_out(verify_shape s, const g1_jac* __restrict__ part, g1_aff* __restrict__ parts,
                                                        size_t nprob) {
  __shared__ fp sm[2 * 128];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = id < nprob * (size_t)s.n_out * 2;
  size_t p = active ? id % nprob : 0;
  size_t r = active ? id / nprob : 0;
  int a = (int)(r & 1), jj = (int)(r >> 1);
  g1_jac acc;
  acc.set_inf();
  if (active) {
    acc = part[((size_t)jj * 2 + a) * nprob + p];
    for (int ch = 1; ch < s.nchunk; ch++) {
      g1_jac t = part[(((size_t)ch * s.n_out + jj) * 2 + a) * nprob + p];
      g1_jac::add(acc, acc, t);
    }
  }
  g1_aff out;
  block_to_affine<128>(out, acc, sm);
  if (active) parts[(p * s.n_out + jj) * 2 + a] = out;
}
// thread -> (p, owned output, a): sum of the `nparts` ranks' partial sums, then the tail of k_vmsm_reduce
__global__ void __launch_bounds__(128) k_vmsm_reduce_parts(verify_shape s, verify_args v, const g1_aff* __restrict__ parts, int nparts,
                                                           g1_aff* __restrict__ X, size_t nprob) {
  __shared__ fp sm[2 * 128];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool active = id < nprob * (size_t)s.n_out_owned() * 2;
  size_t p = active ? id % nprob : 0;
  size_t r = active ? id / nprob : 0;
  int a = (int)(r & 1);
  int jj = active ? s.owned_out((int)(r >> 1)) : 0;
  g1_jac acc;
  acc.set_inf();
  int slot = 0;
  if (active) {
    for (int q = 0; q < nparts; q++) {
      g1_aff t = parts[(((size_t)q * nprob + p) * s.n_out + jj) * 2 + a];
      g1_jac::add_mixed(acc, acc, t);
    }
    if (jj < s.n) {
      slot = jj;
      if (s.groupA && a == 1) {
        g1_aff A = ((const g1_aff*)v.a_consts)[p * s.n + jj];
        g1_jac::add_mixed(acc, acc, A);
      }
    } else if (jj == s.n && !s.groupB) {
      slot = s.sB;
    } else {
      slot = s.sT;
      g1_jac::neg(acc, acc);
    }
  }
  g1_aff out;
  block_to_affine<128>(out, acc, sm);
  if (active) X[((size_t)a * s.K + slot) * nprob + p] = out;
}

// sharded statement: keep the slots k = rank, rank + world, ... (K' of them) of the [2][K][nprob] slot arrays
__global__ void k_gather_owned_slots(const g1_aff* __restrict__ X, const g2_aff* __restrict__ Y, g1_aff* __restrict__ Xo,
                                     g2_aff* __restrict__ Yo, size_t nprob, int K, int Ko, int rank, int world, int do_x,
                                     int do_y) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nprob * (size_t)Ko * 2) return;
  size_t p = id % nprob;
  size_t r = id / nprob;
  int ko = (int)(r % Ko), a = (int)(r / Ko);
  int k = rank + ko * world;
  if (do_x) Xo[((size_t)a * Ko + ko) * nprob + p] = X[((size_t)a * K + k) * nprob + p];
  if (do_y) Yo[((size_t)a * Ko + ko) * nprob + p] = Y[((size_t)a * K + k) * nprob + p];
}
// partial[part][p][e] (AoS, as the ranks exchange them)  ->  F[(part*4 + e)*nprob + p] (launch_final_exp's layout)
__global__ void k_partials_to_chunks(const fp12* __restrict__ partials, fp12* __restrict__ F, size_t nprob, int nparts) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nprob * 4 * (size_t)nparts) return;
  int e = (int)(id & 3);
  size_t p = (id >> 2) % nprob;
  size_t part = (id >> 2) / nprob;
  F[(part * 4 + e) * nprob + p] = partials[id];
}

__global__ void k_and4(const uint8_t* __restrict__ ok4, uint8_t* __restrict__ out, size_t nprob) {
  size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= nprob) return;
  out[p] = ok4[p] & ok4[nprob + p] & ok4[2 * nprob + p] & ok4[3 * nprob + p];
}

// ------------------------------------------------------------------ randomised batch verification (SURVEY.md §8f.4)
// The four ComT entries of every proof p and all proofs of a batch are folded into ONE pairing-product check with random
// weights: entry (a, b) of proof p gets the exponent w_{p,a} * beta_b with (w_{p,0}, w_{p,1}) = (sigma_p, tau_p) drawn per
// proof and (beta_0, beta_1) = (beta, 1) drawn per call, all 64-bit.  By bilinearity the weighted product of the entries is
//     prod_p prod_k e( sigma_p X_k.0 + tau_p X_k.1 ,  beta Y_k.0 + Y_k.1 )      ( = prod_p t_p^tau_p for a PPE )
// over the SAME slots (X_k, Y_k) the exact verifier builds: one Miller pair per slot instead of four (two), and one final
// exponentiation per call instead of four per proof.  Slots whose G2 side is a CRS element share one folded G2 point, so
// their G1 sides are summed over the proofs first.  If any entry of any proof is wrong the check fails except with
// probability <= 2^-62 over the weights (their low 63 bits are used) (a non-zero polynomial of degree 2 in beta, then a non-zero linear form in the
// independent sigma_p, tau_p) -- provided all inputs are in the prime-order groups, as deserialised values are.
// slot_map[k] >= 0: per-proof pair number jw of slot k (G2 side walked); < 0: -(f + 1), CRS slot number f
// resident blocks per SM the fold kernels are compiled for (experiments: -DRFG2_BLOCKS=.. -DRFB_BLOCKS=..)
#ifndef RFG2_BLOCKS
#define RFG2_BLOCKS 2
#endif
#ifndef RFB_BLOCKS
#define RFB_BLOCKS 3
#endif
// sigma x0 + tau x1 by a joint 64-step double-and-add over the table 0, x0, x1, x0 + x1 (one table addition per bit, the
// same instruction stream for every lane; the sum is made affine with one block-wide inversion).  All 128 threads call.
__device__ GS_INL void rand_fold_g1_point(g1_aff& out, const g1_aff& x0, const g1_aff& x1, uint64_t sg, uint64_t tu, fp* sm) {
  g1_aff tab[4];
  tab[0].set_inf();
  tab[1] = x0;
  tab[2] = x1;
  g1_jac j;
  j.from_affine(x0);
  g1_jac::add_mixed(j, j, x1);
  block_to_affine<128>(tab[3], j, sm);
  __syncthreads();  // (sm is reused below)
  g1_jac acc;
  rand_fold_g1_walk(acc, tab, sg, tu);
  block_to_affine<128>(out, acc, sm);
  __syncthreads();
}
// thread -> (p, t), slot k = slot_list[t]:  X' = sigma_p X[0][k][p] + tau_p X[1][k][p]   ->  X1[p*Kw + jw]  |  Xfix[f*nprob + p]
__global__ void __launch_bounds__(128) k_rand_fold_g1(const g1_aff* __restrict__ X, size_t nprob, int K, const uint64_t* __restrict__ rho,
                                                      const int* __restrict__ slot_list, int nlist, const int* __restrict__ slot_map,
                                                      int Kw, g1_aff* __restrict__ X1, g1_aff* __restrict__ Xfix) {
  __shared__ fp sm[2 * 128];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = id < nprob * (size_t)nlist;
  const size_t p = active ? id % nprob : 0;
  const int k = active ? slot_list[id / nprob] : 0;
  g1_aff x0, x1, out;
  x0.set_inf();
  x1.set_inf();
  uint64_t sg = 0, tu = 0;
  if (active) {
    x0 = X[((size_t)0 * K + k) * nprob + p];
    x1 = X[((size_t)1 * K + k) * nprob + p];
    sg = rho[2 * p];
    tu = rho[2 * p + 1];
  }
  rand_fold_g1_point(out, x0, x1, sg, tu, sm);
  if (!active) return;
  const int sm_k = slot_map[k];
  if (sm_k >= 0)
    X1[p * Kw + sm_k] = out;
  else
    Xfix[(size_t)(-sm_k - 1) * nprob + p] = out;
}
// Folded MSM bases (the statement MSM then runs over ONE coordinate, verify_shape::na = 1):
// thread -> (p, q):  q < nbases: xfold[p][q] = sigma_p B_q.0 + tau_p B_q.1 (B_q = c_q, or W1 when A is scalar-valued);
//                    q >= nbases (group-valued A): afold[p][j] = tau_p A_j, j = q - nbases.
// With group-valued B the slot (c_i, iota_2(B_i)) has exactly xfold[p][i] on its G1 side: copied to pair bmap0 + i.
__global__ void __launch_bounds__(128, RFB_BLOCKS) k_rand_fold_bases(verify_shape s, verify_args v, const crs_dev* __restrict__ crs, size_t nprob,
                                                         const uint64_t* __restrict__ rho, g1_aff* __restrict__ xfold,
                                                         g1_aff* __restrict__ afold, int bmap0, int Kw, g1_aff* __restrict__ X1) {
  __shared__ fp sm[2 * 128];
  const int nq = s.nbases + (s.groupA ? s.n : 0);
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = id < nprob * (size_t)nq;
  const size_t p = active ? id % nprob : 0;
  const int q = active ? (int)(id / nprob) : 0;
  g1_aff x0, x1, out;
  x0.set_inf();
  x1.set_inf();
  uint64_t sg = 0, tu = 0;
  if (active) {
    if (q < s.m) {
      x0 = v.xcoms[(p * s.m + q) * 2 + 0];
      x1 = v.xcoms[(p * s.m + q) * 2 + 1];
    } else if (q < s.nbases) {
      x0 = crs->w1[0];
      x1 = crs->w1[1];
    } else {
      x1 = ((const g1_aff*)v.a_consts)[p * s.n + (q - s.nbases)];
    }
    sg = rho[2 * p];
    tu = rho[2 * p + 1];
  }
  rand_fold_g1_point(out, x0, x1, sg, tu, sm);
  if (!active) return;
  if (q < s.nbases) {
    xfold[p * s.nbases + q] = out;
    if (s.groupB && q < s.m) X1[p * Kw + bmap0 + q] = out;
  } else {
    afold[p * s.n + (q - s.nbases)] = out;
  }
}
// thread -> (p, jw): Y' = beta Y[0][k][p] + Y[1][k][p] of slot k = walk_slot[jw]  ->  Y1[p*ostride_p + jw*ostride_j]
// (per-proof pairs: strides (Kw, 1); the pi slots of a big batch, summed over the proofs afterwards: (1, nprob))
__global__ void __launch_bounds__(128, RFG2_BLOCKS) k_rand_fold_g2(const g2_aff* __restrict__ Y, size_t nprob, int K, jsf33 beta,
                                                      const int* __restrict__ walk_slot, int Kw, g2_aff* __restrict__ Y1,
                                                      size_t ostride_p, size_t ostride_j) {
  __shared__ fp sm[2 * 128];
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = id < nprob * (size_t)Kw;
  const size_t p = active ? id % nprob : 0;
  const int jw = active ? (int)(id / nprob) : 0;
  g2_aff y0, y1;
  y0.set_inf();
  y1.set_inf();
  if (active) {
    const int k = walk_slot[jw];
    y0 = Y[((size_t)0 * K + k) * nprob + p];
    y1 = Y[((size_t)1 * K + k) * nprob + p];
  }
  g2_jac acc;
  acc.set_inf();
  const bool any = __syncthreads_or(!y0.is_inf());  // iota_2 images (B_i, a G2 target) have no first coordinate: nothing to fold
  if (any) {
    g2_aff p1, np1, as, ad;
    endo_psi(p1, y0);
    fp2::neg(p1.y, p1.y);  // -psi(Y.0) = |x| Y.0
    np1 = p1;
    fp2::neg(np1.y, p1.y);
    g2_jac js, jd;
    js.from_affine(y0);
    jd = js;
    g2_jac::add_mixed(js, js, p1);
    g2_jac::add_mixed(jd, jd, np1);
    block_to_affine<128>(as, js, sm);
    __syncthreads();
    block_to_affine<128>(ad, jd, sm);
    __syncthreads();
    rand_fold_g2_walk(acc, y0, p1, as, ad, beta);
  }
  g2_jac::add_mixed(acc, acc, y1);
  g2_aff out;
  block_to_affine<128>(out, acc, sm);
  if (active) Y1[p * ostride_p + jw * ostride_j] = out;
}
// thread pid < 3: Yfix[pid] = beta P.0 + P.1 for the CRS elements P = v_1, v_2, W2
__global__ void k_rand_fold_crs(const crs_dev* __restrict__ crs, jsf33 beta, g2_aff* __restrict__ Yfix) {
  const int pid = blockIdx.x * blockDim.x + threadIdx.x;
  if (pid >= 3) return;
  const g2_aff y0 = pid < 2 ? crs->v[pid][0] : crs->w2[0], y1 = pid < 2 ? crs->v[pid][1] : crs->w2[1];
  rand_fold_g2_single(Yfix[pid], y0, y1, beta);
}
// thread -> (f, strip): part[f*nstrips + strip] = sum of L consecutive points of Xfix[f][.]
__global__ void __launch_bounds__(128) k_g1_sum_strips(const g1_aff* __restrict__ Xfix, size_t nprob, int nfix, int L, size_t nstrips,
                                                       g1_jac* __restrict__ part) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (size_t)nfix * nstrips) return;
  const size_t strip = id % nstrips;
  const int f = (int)(id / nstrips);
  g1_jac acc;
  acc.set_inf();
  const size_t p1 = min(nprob, (strip + 1) * L);
  for (size_t p = strip * L; p < p1; p++) g1_jac::add_mixed(acc, acc, Xfix[(size_t)f * nprob + p]);
  part[id] = acc;
}
// block f: X1[at + f] = affine(sum of part[f][.]),  Y1[at + f] = Yfix[fpid[f]]
struct fix_pids {
  int pid[8];
};
__global__ void __launch_bounds__(128) k_g1_sum_final(const g1_jac* __restrict__ part, size_t nstrips, const g2_aff* __restrict__ Yfix,
                                                      fix_pids fp_, size_t at, g1_aff* __restrict__ X1, g2_aff* __restrict__ Y1) {
  __shared__ g1_jac red[128];
  const int f = blockIdx.x, t = threadIdx.x;
  g1_jac acc;
  acc.set_inf();
  for (size_t i = t; i < nstrips; i += 128) {
    g1_jac q = part[(size_t)f * nstrips + i];
    g1_jac::add(acc, acc, q);
  }
  red[t] = acc;
  __syncthreads();
  for (int half = 64; half >= 1; half >>= 1) {
    if (t < half) {
      g1_jac a = red[t], b = red[t + half];
      g1_jac::add(a, a, b);
      red[t] = a;
    }
    __syncthreads();
  }
  if (t == 0) {
    g1_aff o;
    g1_jac::to_affine(o, red[0]);
    X1[at + f] = o;
    Y1[at + f] = Yfix[fp_.pid[f]];
  }
}
__global__ void k_ok1(const uint8_t* __restrict__ ok1, uint8_t* __restrict__ out) { out[0] = ok1[0]; }
// ---- big batches: the slots whose OTHER side is a CRS element are summed over the proofs with the bucket method
// (pippenger.cuh) instead of being folded and paired proof by proof:
//     prod_p e(sigma_p (-u_k.0) + tau_p (-u_k.1), pi'_pk) = e(-u_k.0, sum_p sigma_p pi'_pk) e(-u_k.1, sum_p tau_p pi'_pk)
//     prod_p e(sigma_p th_pk.0 + tau_p th_pk.1, v'_k)     = e(sum_p (sigma_p th_pk.0 + tau_p th_pk.1), v'_k)
// sv[0 .. nprob) = sigma_p, sv[nprob .. 2 nprob) = tau_p as Montgomery Fr values (the scalar format of the MSM kernels)
__global__ void k_rho_to_fr(const uint64_t* __restrict__ rho, size_t nprob, fr* __restrict__ sv) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= 2 * nprob) return;
  const size_t p = id % nprob;
  const uint64_t w = rho[2 * p + (id >= nprob ? 1 : 0)];
  fr x, r2;
  x.set_zero();
  x.l[0] = (uint32_t)w;
  x.l[1] = (uint32_t)(w >> 32);
#pragma unroll
  for (int j = 0; j < 8; j++) r2.l[j] = FR_R2(j);
  fr::mul(x, x, r2);
  sv[id] = x;
}
// pair `at`: ( affine(*sum) , Yfix[pid] )
__global__ void k_rand_place_theta(const g1_jac* __restrict__ sum, const g2_aff* __restrict__ Yfix, int pid, size_t at,
                                   g1_aff* __restrict__ X1, g2_aff* __restrict__ Y1) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  g1_aff o;
  g1_jac::to_affine(o, *sum);
  X1[at] = o;
  Y1[at] = Yfix[pid];
}
// pairs at, at + 1: ( -u_j.row , affine(sums[row * stride]) ), row = 0, 1
__global__ void k_rand_place_pi(const g2_jac* __restrict__ sums, size_t stride, const crs_dev* __restrict__ crs, int j, size_t at,
                                g1_aff* __restrict__ X1, g2_aff* __restrict__ Y1) {
  const int row = threadIdx.x;
  if (row >= 2 || blockIdx.x != 0) return;
  g2_aff o;
  g2_jac::to_affine(o, sums[(size_t)row * stride]);
  X1[at + row] = crs->neg_u[j][row];
  Y1[at + row] = o;
}

// ---- randomised per-proof verification (gs_verify_each_rand): proof p's c accumulators are A = p*c + j; the final
// exponentiation multiplies chunk-major values F[j*nprob + p]
__global__ void k_each_chunk_major(const fp12* __restrict__ M, fp12* __restrict__ F, size_t nprob, int c) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nprob * c) return;
  const size_t p = id % nprob;
  const int j = (int)(id / nprob);
  F[id] = M[p * c + j];
}

// ---- randomised per-statement verification of zk PPEs (gs_zk_ppe_verify_each_rand): statement i's pairs are
// X1 / Y1 [i*Kp + .].  thread -> (i, r): the G1 side of the statement's CRS pair r (0: v_1, 2: W2) gets the folds of its
// K L_k's slots with that CRS point (XfixL[f*nprob*K + i*K + k], lin_pid.pid[f]); pair 0 already holds PPE' theta_0's.
// The threads also copy the L_k's Kl walked pairs (X1L / Y1L [(i*K + k)*Kl + j], j = r/2, r/2 + 2, ...) to pairs
// at_lin + k*Kl + j.  All 128 threads reach the block-wide inversion.
__global__ void __launch_bounds__(128) k_zk_rand_place(size_t nprob, int K, int Kp, int at_lin, const g1_aff* __restrict__ X1L,
                                                       const g2_aff* __restrict__ Y1L, int Kl, const g1_aff* __restrict__ XfixL,
                                                       fix_pids lin_pid, int nfl, g1_aff* __restrict__ X1, g2_aff* __restrict__ Y1) {
  __shared__ fp sm[2 * 128];
  const size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = id < nprob * 2;
  const size_t i = active ? id % nprob : 0;
  const int r = active ? 2 * (int)(id / nprob) : 0;
  g1_jac acc;
  acc.set_inf();
  if (active) {
    const size_t nl = nprob * K;
    if (r == 0) acc.from_affine(X1[i * Kp]);
    for (int k = 0; k < K; k++) {
      const size_t q = i * K + k;
      for (int f = 0; f < nfl; f++)
        if (lin_pid.pid[f] == r) g1_jac::add_mixed(acc, acc, XfixL[f * nl + q]);
      for (int j = r / 2; j < Kl; j += 2) {
        X1[i * Kp + at_lin + k * Kl + j] = X1L[q * Kl + j];
        Y1[i * Kp + at_lin + k * Kl + j] = Y1L[q * Kl + j];
      }
    }
  }
  g1_aff out;
  block_to_affine<128>(out, acc, sm);
  if (active) X1[i * Kp + r] = out;
}

}  // namespace gs


// what the shape alone says about the G2 side of every slot (k_verify_assemble): CRS points have stored lines, iota_2
// images have no first coordinate
static std::vector<uint8_t> slot_kinds(const verify_shape& s) {
  std::vector<uint8_t> kind_all(s.K, gsi::GS_SLOT_WALK);
  for (int k = s.sB; k < s.sPi; k++) kind_all[k] = s.groupB ? gsi::GS_SLOT_WALK_B1 : (uint8_t)(gsi::GS_SLOT_FIXED + 2);
  for (int j = 0; j < s.cy; j++) kind_all[s.sTh + j] = (uint8_t)(gsi::GS_SLOT_FIXED + j);
  if (s.type == 1 || s.type == 3) kind_all[s.sT] = (uint8_t)(gsi::GS_SLOT_FIXED + 2);
  if (s.type == 2) kind_all[s.sT] = gsi::GS_SLOT_WALK_B1;
  return kind_all;
}

// the kinds of the slots k = rank, rank + world, ... that a sharded statement's rank owns
static std::vector<uint8_t> owned_kinds(const std::vector<uint8_t>& kind_all, int rank, int world) {
  std::vector<uint8_t> kind;
  for (size_t k = rank; k < kind_all.size(); k += world) kind.push_back(kind_all[k]);
  return kind;
}

// The G1-side statement MSM of `nprob` problems up to its chunk partials (this rank's bases, s.nb_own(), into the outputs
// it owns): sets s.chunk and s.nchunk, *part = the s.nchunk partial sums.  The caller sums them with its last kernel.
static int statement_msm_partials(gs_ctx* ctx, Scratch& sc, verify_shape& s, const verify_args& v, size_t nprob, bool shared_x,
                                  const g1_jac** part_out) {
  // outputs that share one base coordinate: this rank's MSM outputs x the problems that use the same commitments
  const size_t owned_out = (size_t)s.n_out_owned();
  const size_t na = (size_t)s.na;
  const size_t nb = (size_t)s.nb_own() * na;
  const bool use_wtab = (nprob == 1 || shared_x) && owned_out * nprob >= 320;  // table build ~ 14.6 ms at m = 1024
  {
    // bases per thread: few threads (one statement, or one rank's share of it) -> smaller chunks, so that the
    // grid is ~8 waves of the ~296 resident blocks instead of 1.7 (measured: 20.8 ms for half of C3's sums against
    // 30.8 ms for all of them; C4's shared-table batches 91 -> 67 ms); the table kernel has no doublings to
    // amortise, Straus keeps >= 8.  Many chunks are folded 16 at a time (k_vmsm_fold) before the last kernel.
    int chunk = GS_MSM_CHUNK;
    // (a lone small statement is pure latency: one base per thread there)
    const bool tiny = nprob * owned_out * na * ((s.nb_own() + 7) / 8) < 16384;
    const int floor_chunk = use_wtab ? 4 : (tiny ? 1 : 8);
    while (chunk > floor_chunk && nprob * owned_out * na * ((s.nb_own() + chunk - 1) / chunk) < (size_t)128 * 2368) chunk /= 2;
    set_msm_chunk(s, chunk);
  }
  g1_jac* part;
  CUDA_TRY(sc.alloc(&part, (size_t)s.nchunk * s.n_out * na * nprob));
  if (use_wtab) {
    const wt_geom g = wt_choose(owned_out * nprob);
    const size_t nrows = nb * g.W;
    g1_aff* wtab;
    g1_jac* J;
    CUDA_TRY(sc.alloc(&wtab, nrows * g.H));
    CUDA_TRY(sc.alloc(&J, nrows * g.H));
    LAUNCH(k_wtab_bases, nb, s, v, ctx->crs, J, (int)nb, g);
    LAUNCH(k_jac_to_affine_blocks<1>, nrows, J, wtab, nrows, (size_t)g.H);
    LAUNCH(k_wtab_fill, nrows * (g.H / GS_WT_RUN), wtab, J, nrows, g.H);
    LAUNCH(k_jac_to_affine_blocks<8>, nrows * g.H / 8, J, wtab, nrows * g.H, (size_t)1);
    LAUNCH(k_vmsm_wsum, nprob * owned_out * na * s.nchunk, s, v, wtab, part, nprob, g);
  } else {
    g1_aff* vtab;
    fp* vtabx;
    CUDA_TRY(sc.alloc(&vtab, nb * GS_VTAB * nprob));
    CUDA_TRY(sc.alloc(&vtabx, nb * GS_VTAB * nprob));
    LAUNCH(k_vmsm_tables, nprob * nb, s, v, ctx->crs, vtab, vtabx, nprob);
    LAUNCH(k_vmsm_partial, nprob * owned_out * na * s.nchunk, s, v, vtab, vtabx, part, nprob);
  }
  *part_out = part;
  if (s.nchunk > 32) {  // fold 16 chunks at a time in parallel; the last kernel then walks the few that are left
    const int F = 16, ng = (s.nchunk + F - 1) / F;
    g1_jac* part2;
    CUDA_TRY(sc.alloc(&part2, (size_t)ng * s.n_out * na * nprob));
    LAUNCH(k_vmsm_fold, (size_t)s.n_out * na * nprob * ng, s, part, part2, nprob, s.nchunk, F, ng);
    *part_out = part2;
    s.nchunk = ng;
  }
  return GS_OK;
}

// ---- the eight input arrays of a verify call as one verify_args (host or device addresses)
static verify_args args_of(const void* a_consts, const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                           const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta) {
  verify_args v;
  v.a_consts = a_consts;
  v.b_consts = b_consts;
  v.gamma = (const fr*)gamma;
  v.target = target;
  v.xcoms = (const g1_aff*)xcoms;
  v.ycoms = (const g2_aff*)ycoms;
  v.pi = (const g2_aff*)pi;
  v.theta = (const g1_aff*)theta;
  return v;
}

// the arrays from problem `off` on (Gamma holds s.gm rows per problem)
static verify_args args_at(const verify_shape& s, const verify_args& v, size_t off) {
  verify_args o = v;
  o.a_consts = (const char*)v.a_consts + off * s.n * elem_size_A(s.type);
  o.b_consts = (const char*)v.b_consts + off * s.m * elem_size_B(s.type);
  o.gamma = v.gamma + off * s.gm * s.n;
  o.target = (const char*)v.target + off * elem_size_T(s.type);
  o.xcoms = v.xcoms + off * s.m * 2;
  o.ycoms = v.ycoms + off * s.n * 2;
  o.pi = v.pi + off * s.cx * 2;
  o.theta = v.theta + off * s.cy * 2;
  return o;
}

// device copies of problems [off, off + cnt) of the host arrays `h`, on ctx->stream
static int upload_args(gs_ctx* ctx, Scratch& sc, const verify_shape& s, const verify_args& h, size_t off, size_t cnt, verify_args* d) {
  const verify_args a = args_at(s, h, off);
  uint8_t *dA, *dB, *dT;
  fr* dG;
  g1_aff *dc, *dth;
  g2_aff *dd, *dpi;
  CUDA_TRY(upload(ctx, sc, &dA, a.a_consts, cnt * s.n * elem_size_A(s.type)));
  CUDA_TRY(upload(ctx, sc, &dB, a.b_consts, cnt * s.m * elem_size_B(s.type)));
  CUDA_TRY(upload(ctx, sc, &dG, a.gamma, cnt * s.gm * s.n));
  CUDA_TRY(upload(ctx, sc, &dT, a.target, cnt * elem_size_T(s.type)));
  CUDA_TRY(upload(ctx, sc, &dc, a.xcoms, cnt * s.m * 2));
  CUDA_TRY(upload(ctx, sc, &dd, a.ycoms, cnt * s.n * 2));
  CUDA_TRY(upload(ctx, sc, &dpi, a.pi, cnt * s.cx * 2));
  CUDA_TRY(upload(ctx, sc, &dth, a.theta, cnt * s.cy * 2));
  *d = args_of(dA, dB, (const gs_fr*)dG, dT, (const gs_com1*)dc, (const gs_com2*)dd, (const gs_com2*)dpi, (const gs_com1*)dth);
  return GS_OK;
}

// every input array is set (Gamma may be left out: the rank of gs_verify_sharded that holds no row of it)
static bool inputs_set(const verify_args& v, bool need_gamma = true) {
  return v.a_consts && v.b_consts && (v.gamma || !need_gamma) && v.target && v.xcoms && v.ycoms && v.pi && v.theta;
}

// all `count` rows of `bytes` bytes are equal, count > 1 (equations over ONE set of commitments: a multi-equation statement)
static bool same_rows(const void* rows, size_t count, size_t bytes) {
  for (size_t i = 1; i < count; i++)
    if (memcmp(rows, (const char*)rows + i * bytes, bytes) != 0) return false;
  return count > 1;
}

// ---- argument checks.  Their order decides the code of a call with several bad arguments, and it is not the same for
// every entry point: each one calls these at the point where it has always made that check.
static int check_crs(gs_ctx* ctx) {
  if (!ctx->crs_loaded) FAIL(GS_EARG, "verify: no CRS loaded");
  return GS_OK;
}
// the context, the equation type, the shard (rank, world) and, with `need_crs`, a loaded CRS
static int check_call(gs_ctx* ctx, int type, int rank, int world, bool need_crs) {
  if (!ctx) return GS_EARG;
  if (type < 0 || type > 3) FAIL(GS_EARG, "verify: bad equation type");
  if (world < 1 || rank < 0 || rank >= world) FAIL(GS_EARG, "verify: bad shard (rank, world)");
  return need_crs ? check_crs(ctx) : GS_OK;
}

// a non-empty call: both variable lists non-empty and at most 2^20 long, then all inputs set.  The host front end of
// gs_verify_batch / gs_verify_partial checks its inputs and the CRS ahead of the length limit (`inputs_first`).
static int check_lists(gs_ctx* ctx, size_t m, size_t n, bool inputs, bool inputs_first = false) {
  // the reference panics on empty variable lists (SURVEY.md §3.7): keep it an error
  if (m == 0 || n == 0) FAIL(GS_EDIM, "verify: empty variable list");
  if (inputs_first) {
    if (!inputs) return GS_EARG;
    if (int rc = check_crs(ctx)) return rc;
  }
  if (m > 1 << 20 || n > 1 << 20) FAIL(GS_EDIM, "verify: too many variables");
  return inputs ? GS_OK : GS_EARG;
}

extern "C" {

// Shared body of gs_verify_batch_dev (rank 0 of 1, verdicts) and gs_verify_partial_dev (rank r of w: the
// un-exponentiated Miller products of the slots that rank owns, out_partial[p][4]).  `one_pass`: the caller has cut the
// batch into passes already (verify_host).
static int verify_impl(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const verify_args& args, int rank, int world,
                       uint8_t* out_ok_dev, fp12* out_partial_dev, bool shared_x, bool shared_y = false, bool one_pass = false) {
  if (int rc = check_call(ctx, type, rank, world, true)) return rc;
  if (count == 0) return GS_OK;
  if (int rc = check_lists(ctx, m, n, inputs_set(args))) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  s.rank = rank;
  s.world = world;
  {  // the stored Miller lines of v1, v2, W2 (once per key, on the first verification)
    int rcl = gsi::crs_lines_build(ctx);
    if (rcl) return rcl;
  }
  const int Ko = world > 1 ? (s.K - rank + world - 1) / world : s.K;  // slots this rank owns
  // A batch that needs several passes alternates them between the context's two streams: the passes are independent,
  // so whenever a kernel of one pass leaves SMs idle (the partial last wave of the MSM, a line walk that fills 3/4 of a
  // wave, kernel boundaries) blocks of the other pass take them.  Everything is joined back into gs_stream() at the end.
  const size_t pass_n = verify_pass_size(ctx, count, shared_x, one_pass);
  PassStreams streams(ctx);
  if (count > pass_n && ctx->pass_streams == 2 && !ctx->profile)  // (per-kernel event times need one stream)
    CUDA_TRY(streams.split(true));  // the second stream waits for the inputs (uploaded / produced on the main stream)
  size_t pass = 0;
  for (size_t off = 0; off < count; off += pass_n, pass++) {
    size_t nprob = count - off < pass_n ? count - off : pass_n;
    streams.use(pass);
    Scratch sc(ctx);
    const verify_args v = args_at(s, args, off);
    g1_aff* X;
    g2_aff* Y;
    uint8_t* ok4;
    CUDA_TRY(sc.alloc(&X, 2 * (size_t)s.K * nprob));
    CUDA_TRY(sc.alloc(&Y, 2 * (size_t)s.K * nprob));
    CUDA_TRY(sc.alloc(&ok4, 4 * nprob));
    LAUNCH(k_verify_assemble, nprob * (size_t)s.K, s, v, ctx->crs, X, Y, nprob);
    std::vector<uint8_t> kind_all = slot_kinds(s);
    // equations over ONE set of y-commitments (a multi-equation statement): the (P_j, d_j) slots have the same G2 side in
    // every problem, so lines walked ahead are walked once (C4, 256 PPE equations: 50 k walked points -> 17 k)
    if (shared_y && nprob > 1)
      for (int k = 0; k < s.n; k++) kind_all[k] = gsi::GS_SLOT_WALK_SHARED;
    const std::vector<uint8_t> kind = owned_kinds(kind_all, rank, world);
    // the G2 side is final now: a lone statement starts its line walks on the second stream, next to the MSM below
    g1_aff* Xo = nullptr;
    g2_aff* Yo = nullptr;
    const g2_aff* Yp = Y;
    if (world > 1) {
      CUDA_TRY(sc.alloc(&Xo, 2 * (size_t)(Ko ? Ko : 1) * nprob));
      CUDA_TRY(sc.alloc(&Yo, 2 * (size_t)(Ko ? Ko : 1) * nprob));
      LAUNCH(k_gather_owned_slots, nprob * (size_t)Ko * 2, X, Y, Xo, Yo, nprob, s.K, Ko, rank, world, 0, 1);
      Yp = Yo;
    }
    gsi::walk_ahead wa;  // declared after `sc`: destroyed first, which waits for the walk on every exit path
    if (Ko > 0) {
      int rcw = gsi::g2_walk_ahead(ctx, sc, Yp, nprob, Ko, kind.data(), &wa);
      if (rcw) return rcw;
    }
    {
      const g1_jac* part;
      int rcm = statement_msm_partials(ctx, sc, s, v, nprob, shared_x, &part);
      if (rcm) return rcm;
      LAUNCH(k_vmsm_reduce, nprob * (size_t)s.n_out_owned() * s.na, s, v, part, X, nprob);
    }
    const g1_aff* Xp = X;
    if (world > 1) {
      LAUNCH(k_gather_owned_slots, nprob * (size_t)Ko * 2, X, Y, Xo, Yo, nprob, s.K, Ko, rank, world, 1, 0);
      Xp = Xo;
    }
    int rc;
    if (out_partial_dev) {
      rc = gsi::run_pairing_product(ctx, sc, Xp, Yp, nprob, Ko, nullptr, nullptr, nullptr, out_partial_dev + off * 4, kind.data(), &wa);
      if (rc) return rc;  // (~walk_ahead orders the main stream after the walk before `sc` frees its buffers)
    } else {
      rc = gsi::run_pairing_product(ctx, sc, Xp, Yp, nprob, Ko, nullptr, ok4, type == GS_PPE ? (const fp12*)v.target : nullptr,
                                    nullptr, kind.data(), &wa);
      if (rc) return rc;
      LAUNCH(k_and4, nprob, ok4, out_ok_dev + off, nprob);
    }
  }
  return GS_OK;
}

int gs_verify_batch_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                        const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                        const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, uint8_t* out_ok_dev) {
  if (!out_ok_dev) return GS_EARG;
  return verify_impl(ctx, type, count, m, n, args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta), 0, 1, out_ok_dev,
                     nullptr, false);
}

}  // extern "C"

int gsi::verify_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                    const gs_fr* gamma, const void* target, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                    const gs_com1* theta, bool shared_y, uint8_t* out_ok_dev) {
  return verify_impl(ctx, type, count, m, n, args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta), 0, 1, out_ok_dev,
                     nullptr, false, shared_y);
}

extern "C" {

int gs_verify_partial_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                          const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                          const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, int rank, int world,
                          gs_gt* out_partial_dev) {
  if (!out_partial_dev) return GS_EARG;
  return verify_impl(ctx, type, count, m, n, args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta), rank, world,
                     nullptr, (fp12*)out_partial_dev, false);
}

static int check_finish(gs_ctx* ctx, int type, int nparts) {
  if (int rc = check_call(ctx, type, 0, 1, false)) return rc;
  if (nparts < 1 || nparts > 4096) FAIL(GS_EARG, "verify_finish: bad number of partial products");
  return GS_OK;
}

int gs_verify_finish_dev(gs_ctx* ctx, int type, size_t count, int nparts, const gs_gt* partials_dev, const void* target_dev,
                         uint8_t* out_ok_dev) {
  if (int rc = check_finish(ctx, type, nparts)) return rc;
  if (count == 0) return GS_OK;
  if (!partials_dev || !out_ok_dev || (type == GS_PPE && !target_dev)) return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  fp12* F;
  uint8_t* ok4;
  CUDA_TRY(sc.alloc(&F, (size_t)nparts * 4 * count));
  CUDA_TRY(sc.alloc(&ok4, 4 * count));
  LAUNCH(k_partials_to_chunks, count * 4 * (size_t)nparts, (const fp12*)partials_dev, F, count, nparts);
  int rc = gsi::launch_final_exp(ctx, F, count, nparts, nullptr, ok4, type == GS_PPE ? (const fp12*)target_dev : nullptr);
  if (rc) return rc;
  LAUNCH(k_and4, count, ok4, out_ok_dev, count);
  return GS_OK;
}

// host-buffer front end shared by gs_verify_batch and gs_verify_partial: upload, run, download
static int verify_host(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const verify_args& h, int rank, int world,
                       uint8_t* out_ok, gs_gt* out_partial) {
  if (ctx && count && !out_ok && !out_partial) return GS_EARG;
  if (int rc = check_call(ctx, type, rank, world, false)) return rc;
  if (count == 0) return GS_OK;
  if (int rc = check_lists(ctx, m, n, inputs_set(h), true)) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const verify_shape s = make_verify_shape(type, (int)m, (int)n);
  // a batch of equations over ONE set of x-commitments (a multi-equation statement): detected on the host copy
  const bool shared_x = same_rows(h.xcoms, count, m * sizeof(gs_com1));
  const bool shared_y = same_rows(h.ycoms, count, n * sizeof(gs_com2));
  // Passes of verify_batch_max instances; with two pass streams the H2D copies of pass i + 1 run under the kernels of
  // pass i (pinned host buffers; pageable ones are staged by the driver and serialise on the host side).
  const size_t B = verify_pass_size(ctx, count, shared_x, false);
  const bool pipelined = count > B && ctx->pass_streams == 2 && !ctx->profile && !shared_x;
  const size_t step = pipelined ? B : count;
  {
    PassStreams streams(ctx);
    if (pipelined) CUDA_TRY(streams.split(false));
    size_t pass = 0;
    for (size_t off = 0; off < count; off += step, pass++) {
      const size_t cnt = count - off < step ? count - off : step;
      streams.use(pass);
      Scratch sc(ctx);
      verify_args d;
      uint8_t* dok = nullptr;
      fp12* dpart = nullptr;
      if (int rc = upload_args(ctx, sc, s, h, off, cnt, &d)) return rc;
      if (out_ok)
        CUDA_TRY(sc.alloc(&dok, cnt));
      else
        CUDA_TRY(sc.alloc(&dpart, cnt * 4));
      int rc = verify_impl(ctx, type, cnt, m, n, d, rank, world, dok, dpart, shared_x, shared_y, pipelined);
      if (rc) return rc;
      if (out_ok)
        CUDA_TRY(cudaMemcpyAsync(out_ok + off, dok, cnt, cudaMemcpyDeviceToHost, ctx->stream));
      else
        CUDA_TRY(cudaMemcpyAsync(out_partial + off * 4, dpart, cnt * 4 * sizeof(fp12), cudaMemcpyDeviceToHost, ctx->stream));
    }
  }
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

// ------------------------------------------------------------------ one statement over several GPUs, MSM split by BASE
// gs_verify_partial splits a statement by slot: every rank still needs all m bases for its outputs, so the statement MSM
// (the dominant cost of a big statement, 2 m n scalar products) only shrinks with the number of outputs per rank while
// the shared-base tables do not shrink at all.  Here the MSM is split by BASE instead: rank r builds the tables of the
// bases i = r (mod world) only, sums them into EVERY output, and the partial sums -- n_out x 2 affine G1 points per
// statement -- are exchanged (first all-gather, a real exchange step: every rank needs every other rank's share).  From
// there on the split is by slot as before: rank r adds the partial sums of the outputs it owns, runs its Miller pairs and
// the 4 x 576 B partial products are exchanged (second all-gather); every rank finishes.
// The transport is the caller's (NCCL through torch.distributed, raw NCCL, MPI ...): `allgather(user, send_dev, recv_dev,
// bytes)` must gather `bytes` from every rank into recv_dev (rank-major) and return 0 when recv_dev is complete; both are
// DEVICE pointers and the context's stream is idle while it runs.
static int verify_sharded_impl(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const verify_args& v, int rank, int world,
                               bool shared_x, gs_allgather_fn allgather, void* user, uint8_t* dok) {
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  s.rank = rank;
  s.world = world;
  set_base_shard(s, rank, world);
  {
    int rcl = gsi::crs_lines_build(ctx);
    if (rcl) return rcl;
  }
  const size_t nprob = count;
  if (nprob > ctx->verify_batch_max) FAIL(GS_EDIM, "verify_sharded: too many statements for one pass");
  const int Ko = (s.K - rank + world - 1) / world;  // slots this rank owns
  Scratch sc(ctx);
  // ---- slots, owned G2 side, walk-ahead on the second stream (hidden behind the MSM and the first exchange)
  g1_aff *X, *Xo;
  g2_aff *Y, *Yo;
  CUDA_TRY(sc.alloc(&X, 2 * (size_t)s.K * nprob));
  CUDA_TRY(sc.alloc(&Y, 2 * (size_t)s.K * nprob));
  CUDA_TRY(sc.alloc(&Xo, 2 * (size_t)(Ko ? Ko : 1) * nprob));
  CUDA_TRY(sc.alloc(&Yo, 2 * (size_t)(Ko ? Ko : 1) * nprob));
  LAUNCH(k_verify_assemble, nprob * (size_t)s.K, s, v, ctx->crs, X, Y, nprob);
  const std::vector<uint8_t> kind = owned_kinds(slot_kinds(s), rank, world);
  LAUNCH(k_gather_owned_slots, nprob * (size_t)Ko * 2, X, Y, Xo, Yo, nprob, s.K, Ko, rank, world, 0, 1);
  gsi::walk_ahead wa;  // after `sc`: destroyed first
  if (Ko > 0) {
    int rcw = gsi::g2_walk_ahead(ctx, sc, Yo, nprob, Ko, kind.data(), &wa);
    if (rcw) return rcw;
  }
  // ---- phase A: this rank's bases into EVERY output
  verify_shape sa = s;  // the MSM kernels enumerate outputs through the slot ownership: phase A owns them all
  sa.rank = 0;
  sa.world = 1;
  const size_t all_out = (size_t)sa.n_out;
  g1_aff *myparts, *allparts;
  CUDA_TRY(sc.alloc(&myparts, nprob * all_out * 2));
  CUDA_TRY(sc.alloc(&allparts, (size_t)world * nprob * all_out * 2));
  if (sa.nb_own() > 0) {
    const g1_jac* part;
    int rcm = statement_msm_partials(ctx, sc, sa, v, nprob, shared_x, &part);
    if (rcm) return rcm;
    LAUNCH(k_vmsm_parts_out, nprob * all_out * 2, sa, part, myparts, nprob);
  } else {
    CUDA_TRY(cudaMemsetAsync(myparts, 0, nprob * all_out * 2 * sizeof(g1_aff), ctx->stream));  // no base: identities
  }
  // ---- first exchange: the partial sums
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (allgather(user, myparts, allparts, nprob * all_out * 2 * sizeof(g1_aff)) != 0) FAIL(GS_EARG, "verify_sharded: all-gather of the MSM partial sums failed");
  // ---- phase B: owned outputs -> X slots, owned Miller pairs -> partial products
  LAUNCH(k_vmsm_reduce_parts, nprob * (size_t)s.n_out_owned() * 2, s, v, allparts, world, X, nprob);
  LAUNCH(k_gather_owned_slots, nprob * (size_t)Ko * 2, X, Y, Xo, Yo, nprob, s.K, Ko, rank, world, 1, 0);
  fp12 *mine, *allp;
  CUDA_TRY(sc.alloc(&mine, nprob * 4));
  CUDA_TRY(sc.alloc(&allp, (size_t)world * nprob * 4));
  int rc = gsi::run_pairing_product(ctx, sc, Xo, Yo, nprob, Ko, nullptr, nullptr, nullptr, mine, kind.data(), &wa);
  if (rc) return rc;
  // ---- second exchange: 4 un-exponentiated GT values per statement and rank
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (allgather(user, mine, allp, nprob * 4 * sizeof(fp12)) != 0) FAIL(GS_EARG, "verify_sharded: all-gather of the Miller partial products failed");
  return gs_verify_finish_dev(ctx, type, nprob, world, (const gs_gt*)allp, v.target, dok);
}

int gs_verify_sharded(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                      const gs_fr* gamma_rows, const void* target, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                      const gs_com1* theta, int rank, int world, gs_allgather_fn allgather, void* user, uint8_t* out_ok) {
  const verify_args h = args_of(a_consts, b_consts, gamma_rows, target, xcoms, ycoms, pi, theta);
  if (int rc = check_call(ctx, type, rank, world, true)) return rc;
  if (count == 0) return GS_OK;
  if (int rc = check_lists(ctx, m, n, inputs_set(h, false) && out_ok && allgather)) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  set_base_shard(s, rank, world);
  if (s.gm > 0 && !gamma_rows) return GS_EARG;
  Scratch sc(ctx);
  verify_args d;
  uint8_t* dok;
  if (int rc = upload_args(ctx, sc, s, h, 0, count, &d)) return rc;  // ONLY this rank's rows of Gamma
  CUDA_TRY(sc.alloc(&dok, count));
  int rc = verify_sharded_impl(ctx, type, count, m, n, d, rank, world, same_rows(xcoms, count, m * sizeof(gs_com1)), allgather, user, dok);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(out_ok, dok, count, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

int gs_verify_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                    const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                    const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, uint8_t* out_ok) {
  return verify_host(ctx, type, count, m, n, args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta), 0, 1, out_ok, nullptr);
}

int gs_verify_partial(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                      const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                      const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, int rank, int world,
                      gs_gt* out_partial) {
  return verify_host(ctx, type, count, m, n, args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta), rank, world,
                     nullptr, out_partial);
}

int gs_verify_finish(gs_ctx* ctx, int type, size_t count, int nparts, const gs_gt* partials, const void* target,
                     uint8_t* out_ok) {
  if (int rc = check_finish(ctx, type, nparts)) return rc;
  if (count == 0) return GS_OK;
  if (!partials || !out_ok || (type == GS_PPE && !target)) return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  fp12 *dp, *dT = nullptr;
  uint8_t* dok;
  CUDA_TRY(upload(ctx, sc, &dp, partials, (size_t)nparts * count * 4));
  if (type == GS_PPE) CUDA_TRY(upload(ctx, sc, &dT, target, count));
  CUDA_TRY(sc.alloc(&dok, count));
  int rc = gs_verify_finish_dev(ctx, type, count, nparts, (const gs_gt*)dp, dT, dok);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(out_ok, dok, count, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

}  // extern "C"

// ------------------------------------------------------------------ randomised verification: the stages both drivers share
// Time of a Miller product over `nacc` accumulators of S slots: every accumulator pays 62 squarings (~53 M each as
// executed) next to ~29 M x 68 steps per slot, and the accumulators fill waves of 2 x 148 x 32 lanes
static double acc_cost(size_t nacc, int S) {
  const size_t waves = (nacc + 9471) / 9472;
  return (double)waves * (62.0 * 53.0 + (double)S * 68.0 * 29.0);
}

// The slots of a randomised check: `walk`, whose G2 side is walked proof by proof; `fix`, the CRS slots (G2 side v_1, v_2
// or W2: pid 0, 1, 2); `summed`, summed over the proofs (the bucket sums of the batch check), in neither list.
// k_rand_fold_g1 folds the `all` slots when the statement MSM keeps both coordinates, the `rest` when the commitments are
// folded first.  `map` (where each slot's fold goes) is the driver's encoding; rand_upload makes the device copies.
struct rand_slots {
  std::vector<int> walk, fix, pid, summed, all, rest, map;
  int *dmap = nullptr, *dwalk = nullptr, *dall = nullptr, *drest = nullptr;
};
template <class Summed>
static rand_slots rand_classify(const verify_shape& s, Summed summed) {
  const std::vector<uint8_t> kind = slot_kinds(s);
  rand_slots sl;
  sl.map.assign(s.K, 0);
  for (int k = 0; k < s.K; k++) {
    if (summed(k)) {
      sl.summed.push_back(k);
      continue;
    }
    if (kind[k] >= gsi::GS_SLOT_FIXED) {
      sl.fix.push_back(k);
      sl.pid.push_back(kind[k] - gsi::GS_SLOT_FIXED);
    } else {
      sl.walk.push_back(k);
    }
    // slots whose G1 side k_verify_assemble writes (everything but the MSM outputs); with the commitments folded first the
    // (c_i, iota_2(B_i)) slots need no fold either
    const bool msm_out = k < s.n || (k == s.sB && !s.groupB) || (s.type == 3 && k == s.sT);
    const bool b_slot = s.groupB && k >= s.sB && k < s.sPi;
    sl.all.push_back(k);
    if (!msm_out && !b_slot) sl.rest.push_back(k);
  }
  return sl;
}
static int rand_upload(gs_ctx* ctx, Scratch& top, rand_slots& sl) {
  CUDA_TRY(upload(ctx, top, &sl.dmap, sl.map.data(), sl.map.size()));
  CUDA_TRY(upload(ctx, top, &sl.dwalk, sl.walk.data(), sl.walk.size()));
  CUDA_TRY(upload(ctx, top, &sl.dall, sl.all.data(), sl.all.size()));
  CUDA_TRY(upload(ctx, top, &sl.drest, sl.rest.data(), sl.rest.size()));
  return GS_OK;
}

// beta, the weight of the G2 sides: rho[2 count] in joint sparse form
static jsf33 rand_beta(const uint64_t* rho, size_t count) {
  return make_jsf((uint32_t)rho[2 * count], (uint32_t)(rho[2 * count] >> 32));
}
// the weights (sigma_p, tau_p) of proofs [off, off + nprob) on the device, their low 63 bits: below |x|, so a weight is
// its own first sub-scalar on both groups (bucket sums)
static int rand_weights(gs_ctx* ctx, Scratch& sc, const uint64_t* rho, size_t off, size_t nprob, uint64_t** drho) {
  std::vector<uint64_t> w(rho + 2 * off, rho + 2 * (off + nprob));
  for (uint64_t& x : w) x &= 0x7fffffffffffffffull;
  CUDA_TRY(upload(ctx, sc, drho, w.data(), w.size()));
  return GS_OK;
}

// Proofs per pass: passes of at most `cap` proofs (at most 4 verify_batch_max), equal in size, so that the per-pass
// fixed costs (bucket-sum chains, product trees, partial last waves) are paid as rarely as possible; 0 if `cap` is 0
static size_t rand_pass_size(const gs_ctx* ctx, size_t count, size_t cap) {
  if (cap > 4 * ctx->verify_batch_max) cap = 4 * ctx->verify_batch_max;
  if (ctx->verify_batch_max < 23680) cap = ctx->verify_batch_max;  // (lowered by a test: several passes on a small batch)
  if (cap == 0) return 0;
  const size_t npass = (count + cap - 1) / cap;
  return (count + npass - 1) / npass;
}

// From the assembled slots X / Y [2][K][nprob] to the pairs of the folded problem: the G1 side sigma_p X_k.0 + tau_p X_k.1
// of slot k of proof p goes to X1[p * stride + map[k]] (map[k] < 0: Xfix, the CRS slots of the batch check), the G2 side
// beta Y_k.0 + Y_k.1 of the i-th walked slot to Y1[p * stride + i].  `shared`: one set of commitments under many equations.
static int rand_fold(gs_ctx* ctx, Scratch& sc, verify_shape& s, const verify_args& v, size_t nprob, bool shared, const rand_slots& sl,
                     const uint64_t* drho, const jsf33& beta, g1_aff* X, const g2_aff* Y, int stride, g1_aff* X1, g2_aff* Y1,
                     g1_aff* Xfix) {
  if (!shared) {
    // the commitments are folded BEFORE the statement MSM, which then sums single points: half the scalar products;
    // its outputs are folded slots already, the (c_i, iota_2(B_i)) slots are the folded bases themselves
    g1_aff *xfold, *afold;
    CUDA_TRY(sc.alloc(&xfold, nprob * (size_t)s.nbases));
    CUDA_TRY(sc.alloc(&afold, nprob * (size_t)(s.groupA ? s.n : 1)));
    LAUNCH(k_rand_fold_bases, nprob * (size_t)(s.nbases + (s.groupA ? s.n : 0)), s, v, ctx->crs, nprob, drho, xfold, afold,
           s.groupB ? sl.map[s.sB] : 0, stride, X1);
    verify_shape sf = s;
    sf.na = 1;
    verify_args vf = v;
    vf.xfold = xfold;
    vf.afold = afold;
    vf.fold_map = sl.dmap;
    vf.fold_Kw = stride;
    vf.fold_X1 = X1;
    vf.fold_Xfix = Xfix;
    const g1_jac* part;
    int rcm = statement_msm_partials(ctx, sc, sf, vf, nprob, false, &part);
    if (rcm) return rcm;
    LAUNCH(k_vmsm_reduce, nprob * (size_t)sf.n_out_owned() * sf.na, sf, vf, part, (g1_aff*)nullptr, nprob);
    LAUNCH(k_rand_fold_g1, nprob * sl.rest.size(), X, nprob, s.K, drho, sl.drest, (int)sl.rest.size(), sl.dmap, stride, X1, Xfix);
  } else {
    // the statement MSM keeps its shared-base tables (both coordinates), every slot is folded afterwards
    const g1_jac* part;
    int rcm = statement_msm_partials(ctx, sc, s, v, nprob, true, &part);
    if (rcm) return rcm;
    LAUNCH(k_vmsm_reduce, nprob * (size_t)s.n_out_owned() * s.na, s, v, part, X, nprob);
    LAUNCH(k_rand_fold_g1, nprob * sl.all.size(), X, nprob, s.K, drho, sl.dall, (int)sl.all.size(), sl.dmap, stride, X1, Xfix);
  }
  const int Kw = (int)sl.walk.size();
  LAUNCH(k_rand_fold_g2, nprob * (size_t)Kw, Y, nprob, s.K, beta, sl.dwalk, Kw, Y1, (size_t)stride, (size_t)1);
  return GS_OK;
}

// ------------------------------------------------------------------ randomised batch verification: driver
// slots per Miller accumulator: the multiple of 4 that minimises acc_cost
static int rand_slots_per_acc(size_t npairs) {
  int best = 8;
  double best_t = 1e300;
  for (int S = 8; S <= 128; S += 4) {
    const double t = acc_cost((npairs + S - 1) / S, S);
    if (t < best_t) {
      best_t = t;
      best = S;
    }
  }
  return best;
}

static int verify_rand_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const verify_args& args, const uint64_t* rho_host,
                           bool shared_x, uint8_t* out_ok_dev) {
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  // a big batch sums its pi and theta slots over the proofs with the bucket method (small ones pair them proof by proof:
  // the bucket kernels are dependent chains that do not shrink with the batch)
  const bool use_pip = count >= ctx->rand_pip_min && ctx->verify_batch_max >= 23680;
  rand_slots sl = rand_classify(s, [&](int k) { return use_pip && k >= s.sPi && k < s.sT; });
  const int Kw = (int)sl.walk.size(), nfix = (int)sl.fix.size();
  if (nfix > 8) FAIL(GS_EDIM, "verify_rand: too many CRS slots");
  // per-proof pairs (G2 side walked) at map 0, 1, ..., CRS slots (G1 sides summed over the proofs) at -1, -2, ...
  fix_pids fpids;
  for (int i = 0; i < nfix; i++) {
    sl.map[sl.fix[i]] = -(i + 1);
    fpids.pid[i] = sl.pid[i];
  }
  for (int i = 0; i < Kw; i++) sl.map[sl.walk[i]] = i;
  std::vector<int> pi_slots, theta_slots;
  for (int k : sl.summed) (k < s.sTh ? pi_slots : theta_slots).push_back(k);
  const jsf33 beta = rand_beta(rho_host, count);
  // Passes as large as the line tiles allow (13 KB per pair; half the budget, the slot arrays and tables need room too):
  // 65,536 4x4 PPE proofs are ONE pass.
  size_t pass_n = rand_pass_size(ctx, count, ctx->tile_budget / 2 / 13056 / (size_t)(Kw ? Kw : 1));
  if (pass_n == 0) pass_n = 1;
  const size_t npass = (count + pass_n - 1) / pass_n;
  if ((size_t)pass_n * Kw + nfix > ((size_t)1 << 30)) FAIL(GS_EDIM, "verify_rand: statement too large for one pass");
  Scratch top(ctx);
  fp12 *Mall, *Tall;
  g2_aff* Yfix;
  int* dpi_slots;
  uint8_t* ok1;
  CUDA_TRY(top.alloc(&Mall, npass));
  CUDA_TRY(top.alloc(&Tall, npass + 1));
  CUDA_TRY(top.alloc(&Yfix, 3));
  CUDA_TRY(top.alloc(&ok1, 4));
  if (int rc = rand_upload(ctx, top, sl)) return rc;
  CUDA_TRY(upload(ctx, top, &dpi_slots, pi_slots.data(), pi_slots.size()));
  const bool shared = shared_x && count > 1;
  // The folded CRS points and the target powers prod_p t_p^tau_p depend on nothing the main stream computes: they run on
  // the second stream (latency-bound kernels: a 66-step scalar multiplication in 3 threads, a product tree), next to the
  // statement MSM and the line walk.  (Per-kernel event times need one stream.)
  SideStream side(ctx, !ctx->profile);
  if (int rc = side.fork()) return rc;
  LAUNCH_CFG(k_rand_fold_crs, 3, 32, 0, ctx->crs, beta, Yfix);
  if (int rc = side.back()) return rc;
  size_t pass = 0;
  for (size_t off = 0; off < count; off += pass_n, pass++) {
    const size_t nprob = count - off < pass_n ? count - off : pass_n;
    Scratch sc(ctx);
    SideJoin joined{side};
    const verify_args v = args_at(s, args, off);
    g1_aff *X, *X1, *Xfix;
    g2_aff *Y, *Y1;
    uint64_t* drho;
    if (int rc = rand_weights(ctx, sc, rho_host, off, nprob, &drho)) return rc;
    if (type == GS_PPE) {  // prod_p t_p^tau_p, on the side stream
      if (int rc = side.fork()) return rc;
      fp12* P;
      CUDA_TRY(sc.alloc(&P, nprob));
      int rc = gsi::gt_pow64(ctx, (const fp12*)v.target, drho + 1, 2, nprob, P);
      if (rc) return rc;
      const fp12* Pr = P;
      int nch = (int)nprob;
      rc = gsi::reduce_chunks(ctx, sc, &Pr, 1, &nch, 1, 1);
      if (rc) return rc;
      CUDA_TRY(cudaMemcpyAsync(Tall + pass, Pr, sizeof(fp12), cudaMemcpyDeviceToDevice, ctx->stream));
      if ((rc = side.back())) return rc;
    }
    CUDA_TRY(sc.alloc(&X, 2 * (size_t)s.K * nprob));
    CUDA_TRY(sc.alloc(&Y, 2 * (size_t)s.K * nprob));
    LAUNCH(k_verify_assemble, nprob * (size_t)s.K, s, v, ctx->crs, X, Y, nprob);
    // the folded single-entry problem: nprob * Kw per-proof pairs, then the nfix summed CRS pairs, padded with identities
    const size_t nextra = theta_slots.size() + 2 * pi_slots.size();  // the summed slots: one pair per theta, two per pi
    const size_t npairs = nprob * Kw + nfix + nextra;
    const int S = rand_slots_per_acc(npairs);
    const size_t Ktot = (npairs + S - 1) / S * S;
    CUDA_TRY(sc.alloc(&X1, Ktot));
    CUDA_TRY(sc.alloc(&Y1, Ktot));
    CUDA_TRY(sc.alloc(&Xfix, (size_t)(nfix ? nfix : 1) * nprob));
    CUDA_TRY(cudaMemsetAsync(X1 + npairs, 0, (Ktot - npairs) * sizeof(g1_aff), ctx->stream));
    CUDA_TRY(cudaMemsetAsync(Y1 + npairs, 0, (Ktot - npairs) * sizeof(g2_aff), ctx->stream));
    if (nextra) {
      // bucket sums of the pi / theta slots: they need the assembled slots only, and their kernels are short dependent
      // chains -- on the second stream, next to the statement MSM and the folds
      if (int rc = side.fork()) return rc;
      fr* sv;
      CUDA_TRY(sc.alloc(&sv, 2 * nprob));
      LAUNCH(k_rho_to_fr, 2 * nprob, drho, nprob, sv);
      size_t at = nprob * Kw + nfix;
      for (size_t t = 0; t < theta_slots.size(); t++, at++) {
        const int k = theta_slots[t];  // (theta slot sTh + j pairs with the CRS point j)
        g1_jac* sum;
        size_t stride;
        int rcp = gsi::pippenger_rows<FpOps>(ctx, sc, sv, 1, X + ((size_t)0 * s.K + k) * nprob, nprob, X + ((size_t)1 * s.K + k) * nprob,
                                              nprob, &sum, &stride, 0, 63);
        if (rcp) return rcp;
        LAUNCH_CFG(k_rand_place_theta, 1, 32, 0, sum, Yfix, k - s.sTh, at, X1, Y1);
      }
      if (!pi_slots.empty()) {
        g2_aff* Ypi;
        CUDA_TRY(sc.alloc(&Ypi, pi_slots.size() * nprob));
        LAUNCH(k_rand_fold_g2, nprob * pi_slots.size(), Y, nprob, s.K, beta, dpi_slots, (int)pi_slots.size(), Ypi, (size_t)1, nprob);
        for (size_t t = 0; t < pi_slots.size(); t++, at += 2) {
          g2_jac* sums;
          size_t stride;
          int rcp = gsi::pippenger_rows<Fp2Ops>(ctx, sc, sv, 2, Ypi + t * nprob, nprob, (const g2_aff*)nullptr, 0, &sums, &stride, 0, 63);
          if (rcp) return rcp;
          LAUNCH_CFG(k_rand_place_pi, 32, 32, 0, sums, stride, ctx->crs, pi_slots[t] - s.sPi, at, X1, Y1);
        }
      }
      if (int rc = side.back()) return rc;
    }
    if (int rc = rand_fold(ctx, sc, s, v, nprob, shared, sl, drho, beta, X, Y, Kw, X1, Y1, Xfix)) return rc;
    if (int rc = side.join()) return rc;  // the folded CRS points (and, long finished, this pass's target powers)
    if (nfix) {
      const int L = 32;
      const size_t nstrips = (nprob + L - 1) / L;
      g1_jac* part;
      CUDA_TRY(sc.alloc(&part, (size_t)nfix * nstrips));
      LAUNCH(k_g1_sum_strips, (size_t)nfix * nstrips, Xfix, nprob, nfix, L, nstrips, part);
      LAUNCH_CFG(k_g1_sum_final, (size_t)nfix * 128, 128, 0, part, nstrips, Yfix, fpids, nprob * Kw, X1, Y1);
    }
    int rc = gsi::run_pairing_product(ctx, sc, X1, Y1, 1, (int)Ktot, nullptr, nullptr, nullptr, Mall + pass, nullptr, nullptr, 1, S);
    if (rc) return rc;
  }
  const fp12* want = nullptr;
  if (type == GS_PPE) {
    const fp12* Tr = Tall;
    int nch = (int)npass;
    Scratch sc(ctx);
    int rc = gsi::reduce_chunks(ctx, sc, &Tr, 1, &nch, 1, 1);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(Tall + npass, Tr, sizeof(fp12), cudaMemcpyDeviceToDevice, ctx->stream));
    want = Tall + npass;
  }
  int rc = gsi::launch_final_exp(ctx, Mall, 1, (int)npass, nullptr, ok1, want, 1);
  if (rc) return rc;
  LAUNCH_CFG(k_ok1, 1, 32, 0, ok1, out_ok_dev);
  return GS_OK;
}

// ------------------------------------------------------------------ randomised per-proof verification: driver
// The fold of verify_rand_dev stopped one step early: the four ComT entries of proof p are folded with ITS weights
// (sigma_p, tau_p) and the call's beta, and nothing is multiplied across proofs.  Proof p is accepted iff
//     FE( prod_k e( sigma_p X_k.0 + tau_p X_k.1 ,  beta Y_k.0 + Y_k.1 ) )  ==  t_p^tau_p   (PPE; 1 for the other types)
// over the slots (X_k, Y_k) of the exact verifier.  A proof that fails the exact check has a non-zero 2 x 2 matrix E of
// exponent errors and passes only if sigma beta E00 + sigma E01 + tau beta E10 + tau E11 = 0, a non-zero polynomial of
// degree 2 in (sigma_p, tau_p, beta): probability <= 2^-62 over 63-bit weights, for every proof on its own (beta being
// shared does not matter).  Preconditions as for the batch check.
// Pairs of proof p, contiguous: X1 / Y1 [p*Kp + i], i < nf: the CRS slots (G2 side = one of the three folded CRS points,
// lines walked once per call, Y1 left the identity), then the Kw walked slots, then identity padding.  Proof p takes the c
// accumulators p*c .. p*c + c - 1 of S slots each (Kp = c S); c = 1 unless the proofs are few or large.
static void each_split(size_t nprob, int Kp0, int* S_out, int* c_out) {
  // at most M4_MAXS = 512 slots per accumulator
  int best_S = 0, best_c = 1;
  double best_t = 1e300;
  for (int c = 1; c <= Kp0; c++) {
    const int S = ((Kp0 + c - 1) / c + 3) / 4 * 4;
    if (S > 512) continue;
    if (S < 8 && c > 1) break;
    const double t = acc_cost(nprob * c, S);
    if (t < best_t) {
      best_t = t;
      best_S = S;
      best_c = c;
    }
  }
  *S_out = best_S;
  *c_out = best_c;
}

// The folded CRS points of beta (Yfix, 3 of them, owned by `top`) and their lines, on the side stream
static int each_crs_points(gs_ctx* ctx, Scratch& top, SideStream& side, const jsf33& beta, g2_aff** Yfix, fp2** lines) {
  CUDA_TRY(top.alloc(Yfix, 3));
  if (int rc = side.fork()) return rc;
  LAUNCH_CFG(k_rand_fold_crs, 3, 32, 0, ctx->crs, beta, *Yfix);
  if (int rc = gsi::g2_lines(ctx, top, *Yfix, 3, lines)) return rc;
  return side.back();
}

// The Miller products of a pass of nprob proofs (c accumulators of S pairs each, `each`), their final exponentiations and
// the verdicts out_ok_dev[p] = (FE(product of proof p) == want[p]) (want null: 1)
static int each_finish(gs_ctx* ctx, Scratch& sc, const g1_aff* X1, const g2_aff* Y1, size_t nprob, int S, int c, gsi::acc_each& each,
                       const fp12* want, uint8_t* out_ok_dev) {
  fp12* M;
  CUDA_TRY(sc.alloc(&M, nprob * (size_t)c));
  each.F = M;
  int rc = gsi::run_pairing_product(ctx, sc, X1, Y1, 1, (int)(nprob * (size_t)S * c), nullptr, nullptr, nullptr, nullptr, nullptr,
                                    nullptr, 1, S, &each);
  if (rc) return rc;
  const fp12* Fr = M;
  int nch = c;
  if (c > 1) {
    fp12* F;
    CUDA_TRY(sc.alloc(&F, nprob * (size_t)c));
    LAUNCH(k_each_chunk_major, nprob * (size_t)c, M, F, nprob, c);
    Fr = F;
    if (nch > 12) {
      rc = gsi::reduce_chunks(ctx, sc, &Fr, nprob, &nch, 12, 1);
      if (rc) return rc;
    }
  }
  return gsi::launch_final_exp(ctx, Fr, nprob, nch, nullptr, out_ok_dev, want, 1);
}

static int verify_each_rand_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const verify_args& args,
                                const uint64_t* rho_host, bool shared_x, uint8_t* out_ok_dev) {
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  rand_slots sl = rand_classify(s, [](int) { return false; });
  const int Kw = (int)sl.walk.size(), nf = (int)sl.fix.size();
  if (nf > 4) FAIL(GS_EDIM, "verify_each_rand: too many CRS slots");
  gsi::acc_each each;
  each.nf = nf;
  for (int i = 0; i < nf; i++) {
    sl.map[sl.fix[i]] = i;
    each.pid[i] = sl.pid[i];
  }
  for (int i = 0; i < Kw; i++) sl.map[sl.walk[i]] = nf + i;
  const jsf33 beta = rand_beta(rho_host, count);
  // Passes as large as the line tiles allow (13,056 B per pair), equal in size.  Unlike verify_rand_dev the whole tile
  // budget goes to the tiles: a per-proof pass has no bucket sums or product trees beside them, and 65,536 4x4 PPE proofs
  // (12 pairs each) then run as one pass of 6.9 waves instead of two of 3.5 (4 + 4 waves of k_miller4).
  int S, c;
  each_split(count, nf + Kw, &S, &c);
  if (S == 0) FAIL(GS_EDIM, "verify_each_rand: statement too large");
  const int Kp = S * c;
  const size_t pass_n = rand_pass_size(ctx, count, ctx->tile_budget / 13056 / (size_t)Kp);
  if (pass_n == 0) FAIL(GS_EDIM, "verify_each_rand: one proof exceeds the tile budget");
  if (pass_n * (size_t)Kp > ((size_t)1 << 30)) FAIL(GS_EDIM, "verify_each_rand: statement too large for one pass");
  Scratch top(ctx);
  if (int rc = rand_upload(ctx, top, sl)) return rc;
  const bool shared = shared_x && count > 1;
  // The folded CRS points, their lines and the target powers t_p^tau_p depend on nothing the main stream computes: they
  // run on the second stream, next to the statement MSM and the folds.
  SideStream side(ctx, !ctx->profile);
  g2_aff* Yfix = nullptr;
  fp2* crs_lines = nullptr;
  if (nf)
    if (int rc = each_crs_points(ctx, top, side, beta, &Yfix, &crs_lines)) return rc;
  each.pts = Yfix;
  each.lines = crs_lines;
  each.acc_stride = c;
  for (size_t off = 0; off < count; off += pass_n) {
    const size_t nprob = count - off < pass_n ? count - off : pass_n;
    Scratch sc(ctx);
    SideJoin joined{side};
    const verify_args v = args_at(s, args, off);
    g1_aff *X, *X1;
    g2_aff *Y, *Y1;
    uint64_t* drho;
    fp12* want = nullptr;
    if (int rc = rand_weights(ctx, sc, rho_host, off, nprob, &drho)) return rc;
    if (type == GS_PPE) {  // t_p^tau_p, on the side stream
      CUDA_TRY(sc.alloc(&want, nprob));
      if (int rc = side.fork()) return rc;
      if (int rc = gsi::gt_pow64(ctx, (const fp12*)v.target, drho + 1, 2, nprob, want)) return rc;
      if (int rc = side.back()) return rc;
    }
    const size_t Ktot = nprob * (size_t)Kp;
    CUDA_TRY(sc.alloc(&X, 2 * (size_t)s.K * nprob));
    CUDA_TRY(sc.alloc(&Y, 2 * (size_t)s.K * nprob));
    CUDA_TRY(sc.alloc(&X1, Ktot));
    CUDA_TRY(sc.alloc(&Y1, Ktot));
    CUDA_TRY(cudaMemsetAsync(X1, 0, Ktot * sizeof(g1_aff), ctx->stream));  // padding and the CRS pairs' G2 sides: identities
    CUDA_TRY(cudaMemsetAsync(Y1, 0, Ktot * sizeof(g2_aff), ctx->stream));
    LAUNCH(k_verify_assemble, nprob * (size_t)s.K, s, v, ctx->crs, X, Y, nprob);
    if (int rc = rand_fold(ctx, sc, s, v, nprob, shared, sl, drho, beta, X, Y, Kp, X1, Y1 + nf, nullptr)) return rc;
    if (int rc = side.join()) return rc;  // the folded CRS points and their lines, this pass's target powers
    if (int rc = each_finish(ctx, sc, X1, Y1, nprob, S, c, each, want, out_ok_dev + off)) return rc;
  }
  return GS_OK;
}

// ------------------------------------------------------------------ randomised per-statement verification of zk PPEs
// (gs_zk_ppe_verify_each_rand).  Statement i is PPE' (target 1) and its K equations L_k (target O, iota_T(O) = 1).  Every
// equation e has weights of its own, (sigma_e, tau_e), the call one beta; each equation's slots are folded as
// verify_each_rand_dev folds them, and all folded pairs of the statement go into ONE Miller product:
//     accept i  iff  FE( prod_e prod_k e( sigma_e X_k.0 + tau_e X_k.1 ,  beta Y_k.0 + Y_k.1 ) ) == 1.
// A statement the exact verifier rejects has some equation with a non-zero error matrix E^(e) and passes only if
// sum_e (sigma_e beta E00 + sigma_e E01 + tau_e beta E10 + tau_e E11) = 0: a non-zero polynomial of degree 2, probability
// <= 2^-62 over 63-bit weights.  The weights must be independent per equation: with shared ones, errors +D on PPE' theta_0
// and -D on L_k's theta (both paired with v_1) cancel.
// By bilinearity every slot of the statement whose G2 side is the same CRS point becomes ONE pair (the G1 sides summed):
// statement i's pairs are [i*Kp + .] = (v_1: PPE' theta_0 + the L_k's theta), (v_2: PPE' theta_1), (W2: the L_k's d, b c
// and target slots), then PPE''s walked slots, then the two walked pi slots of every L_k, then identity padding.  At
// m = n = 4, K = 1 that is 3 + 13 = 16 pairs, one accumulator.  L_k's d-slot, which slot_kinds marks walked, is W2 here.
int gsi::zk_each_rand_dev(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts, const gs_g2* b_consts,
                          const gs_fr* gamma, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta,
                          const gs_g1* lin_a, const gs_fr* lin_b, const gs_fr* lin_gamma, const gs_g1* lin_target,
                          const gs_com1* lin_xcoms, const gs_com2* lin_ycoms, const gs_com2* lin_pi, const gs_com1* lin_theta,
                          const uint64_t* rho_ppe, const uint64_t* rho_lin, const uint64_t* rho_beta, uint8_t* out_ok_dev) {
  verify_shape sp = make_verify_shape(GS_PPE, (int)m, (int)n), sl = make_verify_shape(GS_MSMEG1, 1, 1);
  const verify_args ap = args_of(a_consts, b_consts, gamma, nullptr, xcoms, ycoms, pi, theta);
  const verify_args al = args_of(lin_a, lin_b, lin_gamma, lin_target, lin_xcoms, lin_ycoms, lin_pi, lin_theta);
  constexpr int nf = 3;  // the CRS pairs, pid 0, 1, 2
  // PPE': theta_j (CRS pid j) folds straight into pair j, the walked slots into pairs nf, nf + 1, ...
  rand_slots slp = rand_classify(sp, [](int) { return false; });
  const int KwP = (int)slp.walk.size();
  for (size_t f = 0; f < slp.fix.size(); f++) slp.map[slp.fix[f]] = slp.pid[f];
  for (int i = 0; i < KwP; i++) slp.map[slp.walk[i]] = nf + i;
  // L_k: the d-slot joins the W2 slots; all CRS slots to XfixL (-1, -2, ...), the walked pi slots to pairs 0, 1 of its own
  rand_slots sll = rand_classify(sl, [](int) { return false; });
  sll.walk.erase(std::find(sll.walk.begin(), sll.walk.end(), 0));
  sll.fix.push_back(0);
  sll.pid.push_back(2);
  const int Kl = (int)sll.walk.size(), nfl = (int)sll.fix.size();
  fix_pids lin_pid;
  for (int f = 0; f < nfl; f++) {
    sll.map[sll.fix[f]] = -(f + 1);
    lin_pid.pid[f] = sll.pid[f];
  }
  for (int i = 0; i < Kl; i++) sll.map[sll.walk[i]] = i;
  gsi::acc_each each;
  each.nf = nf;
  for (int f = 0; f < nf; f++) each.pid[f] = f;
  const jsf33 beta = rand_beta(rho_beta, 0);
  const size_t at_lin = nf + (size_t)KwP, Kpair = at_lin + K * (size_t)Kl;
  int S, c;
  each_split(count, (int)Kpair, &S, &c);
  if (S == 0) FAIL(GS_EDIM, "zk_ppe_verify_each_rand: statement too large");
  const int Kp = S * c;
  const size_t pass_n = rand_pass_size(ctx, count, ctx->tile_budget / 13056 / (size_t)Kp);
  if (pass_n == 0) FAIL(GS_EDIM, "zk_ppe_verify_each_rand: one statement exceeds the tile budget");
  if (pass_n * (size_t)Kp > ((size_t)1 << 30)) FAIL(GS_EDIM, "zk_ppe_verify_each_rand: statement too large for one pass");
  Scratch top(ctx);
  if (int rc = rand_upload(ctx, top, slp)) return rc;
  if (int rc = rand_upload(ctx, top, sll)) return rc;
  SideStream side(ctx, !ctx->profile);
  g2_aff* Yfix;
  fp2* crs_lines;
  if (int rc = each_crs_points(ctx, top, side, beta, &Yfix, &crs_lines)) return rc;
  each.pts = Yfix;
  each.lines = crs_lines;
  each.acc_stride = c;
  for (size_t off = 0; off < count; off += pass_n) {
    const size_t nprob = count - off < pass_n ? count - off : pass_n, nl = nprob * K;
    Scratch sc(ctx);
    SideJoin joined{side};
    const verify_args vp = args_at(sp, ap, off), vl = args_at(sl, al, off * K);
    g1_aff *XP, *XL, *X1, *X1L, *XfixL;
    g2_aff *YP, *YL, *Y1, *Y1L;
    uint64_t *drp, *drl;
    if (int rc = rand_weights(ctx, sc, rho_ppe, off, nprob, &drp)) return rc;
    if (int rc = rand_weights(ctx, sc, rho_lin, off * K, nl, &drl)) return rc;
    const size_t Ktot = nprob * (size_t)Kp;
    CUDA_TRY(sc.alloc(&XP, 2 * (size_t)sp.K * nprob));
    CUDA_TRY(sc.alloc(&YP, 2 * (size_t)sp.K * nprob));
    CUDA_TRY(sc.alloc(&XL, 2 * (size_t)sl.K * nl));
    CUDA_TRY(sc.alloc(&YL, 2 * (size_t)sl.K * nl));
    CUDA_TRY(sc.alloc(&X1, Ktot));
    CUDA_TRY(sc.alloc(&Y1, Ktot));
    CUDA_TRY(sc.alloc(&X1L, nl * Kl));
    CUDA_TRY(sc.alloc(&Y1L, nl * Kl));
    CUDA_TRY(sc.alloc(&XfixL, nl * nfl));
    CUDA_TRY(cudaMemsetAsync(X1, 0, Ktot * sizeof(g1_aff), ctx->stream));  // padding and the CRS pairs' G2 sides: identities
    CUDA_TRY(cudaMemsetAsync(Y1, 0, Ktot * sizeof(g2_aff), ctx->stream));
    LAUNCH(k_verify_assemble, nprob * (size_t)sp.K, sp, vp, ctx->crs, XP, YP, nprob);
    LAUNCH(k_verify_assemble, nl * (size_t)sl.K, sl, vl, ctx->crs, XL, YL, nl);
    if (int rc = rand_fold(ctx, sc, sp, vp, nprob, false, slp, drp, beta, XP, YP, Kp, X1, Y1 + nf, nullptr)) return rc;
    if (int rc = rand_fold(ctx, sc, sl, vl, nl, false, sll, drl, beta, XL, YL, Kl, X1L, Y1L, XfixL)) return rc;
    LAUNCH(k_zk_rand_place, nprob * 2, nprob, (int)K, Kp, (int)at_lin, X1L, Y1L, Kl, XfixL, lin_pid, nfl, X1, Y1);
    if (int rc = side.join()) return rc;  // the folded CRS points and their lines
    if (int rc = each_finish(ctx, sc, X1, Y1, nprob, S, c, each, nullptr, out_ok_dev + off)) return rc;
  }
  return GS_OK;
}

// gs_verify_batch_rand / gs_verify_each_rand past their checks: the host arrays uploaded, the driver, `nout` verdict bytes
// copied back
static int rand_host(gs_ctx* ctx, decltype(&verify_rand_dev) driver, int type, size_t count, size_t m, size_t n, const verify_args& h,
                     const uint64_t* rho, uint8_t* out, size_t nout) {
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  verify_args d;
  uint8_t* dok;
  if (int rc = upload_args(ctx, sc, make_verify_shape(type, (int)m, (int)n), h, 0, count, &d)) return rc;
  CUDA_TRY(sc.alloc(&dok, nout));
  int rc = driver(ctx, type, count, m, n, d, rho, same_rows(h.xcoms, count, m * sizeof(gs_com1)), dok);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, dok, nout, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

extern "C" {

int gs_verify_batch_rand(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                         const gs_fr* gamma, const void* target, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                         const gs_com1* theta, const uint64_t* rho, uint8_t* out_all_ok) {
  const verify_args h = args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta);
  if (int rc = check_call(ctx, type, 0, 1, true)) return rc;
  if (!out_all_ok) return GS_EARG;
  if (count == 0) {
    *out_all_ok = 1;
    return GS_OK;
  }
  if (int rc = check_lists(ctx, m, n, inputs_set(h) && rho)) return rc;
  return rand_host(ctx, verify_rand_dev, type, count, m, n, h, rho, out_all_ok, 1);
}

int gs_verify_batch_rand_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                             const gs_fr* gamma, const void* target, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                             const gs_com1* theta, const uint64_t* rho, uint8_t* out_all_ok_dev) {
  const verify_args v = args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta);
  if (int rc = check_call(ctx, type, 0, 1, true)) return rc;
  if (count == 0 || !out_all_ok_dev) return GS_EARG;
  if (int rc = check_lists(ctx, m, n, inputs_set(v) && rho)) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  return verify_rand_dev(ctx, type, count, m, n, v, rho, false, out_all_ok_dev);
}

int gs_verify_each_rand(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                        const gs_fr* gamma, const void* target, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                        const gs_com1* theta, const uint64_t* rho, uint8_t* out_ok) {
  const verify_args h = args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta);
  if (int rc = check_call(ctx, type, 0, 1, true)) return rc;
  if (count == 0) return GS_OK;
  if (!out_ok) return GS_EARG;
  if (int rc = check_lists(ctx, m, n, inputs_set(h) && rho)) return rc;
  return rand_host(ctx, verify_each_rand_dev, type, count, m, n, h, rho, out_ok, count);
}

int gs_verify_each_rand_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                            const gs_fr* gamma, const void* target, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                            const gs_com1* theta, const uint64_t* rho, uint8_t* out_ok_dev) {
  const verify_args v = args_of(a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta);
  if (int rc = check_call(ctx, type, 0, 1, true)) return rc;
  if (count == 0) return GS_OK;
  if (!out_ok_dev) return GS_EARG;
  if (int rc = check_lists(ctx, m, n, inputs_set(v) && rho)) return rc;
  CUDA_TRY(cudaSetDevice(ctx->device));
  return verify_each_rand_dev(ctx, type, count, m, n, v, rho, false, out_ok_dev);
}

}  // extern "C"
