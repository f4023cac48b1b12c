// Pairing-product pipeline: G2 line preparation, Miller accumulation, final exponentiation, and the
// ComT entry points of the C ABI (ComT::pairing / pairing_sum / linear_map_*, E::pairing).
// Reference: src/data_structures.rs:484-540, src/generator.rs:116.
#include "ctx.h"
#include "batchinv.cuh"
#include "coop12.cuh"
#include "pairing.cuh"

using namespace gs;

namespace gs {

// "Slot" layout used by every pairing-product evaluation (ComT::pairing, pairing_sum, verify): a problem
// is K pairs (X_k in Com1, Y_k in Com2), and the wanted ComT is
//     ComT[a][b] = prod_k e(X_k.a, Y_k.b)          (src/data_structures.rs:494-502)
// Points are stored SoA over problems so that a warp (32 consecutive problems, same slot, same
// coordinate) reads contiguous memory:
//     X[(a*K + k) * nprob + p]   g1_aff        Y[(b*K + k) * nprob + p]   g2_aff

// ------------------------------------------------------------------ evaluated line tiles + cooperative Miller
// Accumulator index A = chunk * np + (p - p0) (chunk = slot range [chunk*S, chunk*S+S) of a big statement);
// 32 consecutive accumulators of one ComT entry e = 2a+b form a block  bid = (A/32)*4 + e.
// Tile (bid, kk, step): the line of slot kk at Miller step `step`, evaluated at the G1 point of entry e and
// scaled so that its w^3 coefficient is one:  l' = w^3 + beta w^2 + alpha  with  beta = lam * (-xP/yP),
// alpha = mu / yP  (pairing.cuh g2_affine_step).  Stored as 4 Fp (alpha.c0 alpha.c1 beta.c0 beta.c1) in the
// Q layout of coop12.cuh, 6,144 B, contiguous: written by k_g2_prepare4 with 16-B stores (512 B per warp
// and quad), copied into shared memory by k_miller4 with cp.async.
//     tiles[((bid*S + kk)*68 + step) * M4_TILE ...]      masks[bid*S + kk] = lanes whose pair is not dropped
constexpr int M4_NV = 4;
constexpr int M4_TILE = M4_NV * CQ_FP;
constexpr int M4_MAXS = 512;
constexpr int M4_SMEM = (2 * CQ_ACC + 2 * M4_TILE) * 4 + M4_MAXS * 6 + 16;  // per 6-warp group

// per G1 slot point: PW[((a*K + k)*2 + which)*12 + limb][pl] with which = 0: -xP/yP, 1: 1/yP (zero for identity)
__global__ void __launch_bounds__(128) k_g1_prep(const g1_aff* __restrict__ X, uint32_t* __restrict__ PW, size_t nprob,
                                                 size_t p0, size_t np, int K, int na) {
  __shared__ fp sm[2 * 128];
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  bool in = q < (size_t)na * K * np;
  size_t pl = in ? q % np : 0, ak = in ? q / np : 0;
  fp x, w;
  x.set_zero();
  w.set_zero();
  if (in) {
    const g1_aff* P = &X[ak * nprob + p0 + pl];
    x = P->x;
    w = P->y;
    if (x.is_zero() && w.is_zero()) w.set_zero();
  }
  block_batch_inv<128>(w, sm);  // 0 stays 0
  if (!in) return;
  fp s;
  fp::mul(s, x, w);
  fp::neg(s, s);
  uint32_t* o = PW + (ak * 2 * 12) * np + pl;
#pragma unroll
  for (int j = 0; j < 12; j++) {
    o[(size_t)j * np] = s.l[j];
    o[(size_t)(12 + j) * np] = w.l[j];
  }
}

// k_g2_prepare4<E>: one thread per (group of E walk-list entries, problem).  The E running points T_i (192 B each)
// live in thread-local memory (L1/L2-resident, lane-interleaved by the hardware): shared memory would cap the
// kernel at 8 warps per SM, and the walk is latency-bound (long dependent chains in the division steps), so
// occupancy matters more than the few hundred bytes of local traffic per step (20 warps/SM at 96 registers).
// tile stores bypass the usual L2 retention (st.global.cs): the tiles are written once and read once by k_miller4
// much later, while the running points in local memory should stay L2-resident.
__device__ GS_INL void cq_st_stream(uint32_t* p, const fp& a) {
#pragma unroll
  for (int q = 0; q < 3; q++)
    __stcs((uint4*)(p + q * CQ_QUAD), make_uint4(a.l[q * 4], a.l[q * 4 + 1], a.l[q * 4 + 2], a.l[q * 4 + 3]));
}
// walk[e] = (b << 31) | k: the (coordinate, slot) pairs that have a G2 point to walk, packed so that every thread's E
// points exist (slots known to be iota_2 images contribute only b = 1, CRS slots none: k_fixed_tiles serves them).
struct g2_pts_list {  // the fixed points Q_i of one thread (read again at the 5 addition steps only)
  const g2_aff* q[8];
  __device__ GS_INL void ld(int i, fp2& X, fp2& Y) const {
    X = q[i]->x;
    Y = q[i]->y;
  }
};
template <int E, int MINB>
__global__ void __launch_bounds__(128, MINB) k_g2_prepare4(const uint32_t* __restrict__ PW, const g2_aff* __restrict__ Y,
                                                        uint32_t* __restrict__ tiles, uint32_t* __restrict__ masks,
                                                        size_t nprob, size_t p0, size_t np, int K, int S,
                                                        const uint32_t* __restrict__ walk, int nwalk, int ne) {
  const int G = (nwalk + E - 1) / E;
  const int na = ne == 4 ? 2 : 1;  // ne = 1: single-entry products (one G1 and one G2 coordinate per slot)
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool inrange = q < (size_t)G * np;
  if (!inrange) q = 0;
  const size_t pl = q % np;
  const int g = (int)(q / np);
  fp2 Tx[E], Ty[E];
  g2_pts_arr T{Tx, Ty};
  g2_pts_list Q;
  bool act[E], acta[E][2];
  size_t tb[E][2];
  int lanes[E], kslot[E];
  bool any = false;
#pragma unroll
  for (int i = 0; i < E; i++) {
    const int e = g * E + i;
    act[i] = false;
    acta[i][0] = acta[i][1] = false;
    tb[i][0] = tb[i][1] = 0;
    lanes[i] = 0;
    kslot[i] = 0;
    Q.q[i] = Y;
    if (e >= nwalk || !inrange) continue;
    const uint32_t we = walk[e];
    const int b = (int)(we >> 31), k = (int)(we & 0x3FFFFFFFu);
    kslot[i] = k;
    Q.q[i] = &Y[((size_t)b * K + k) * nprob + p0 + pl];
    fp2 qx, qy;
    Q.ld(i, qx, qy);
    if (qx.is_zero() && qy.is_zero()) continue;
    const int ch = k / S, kk = k % S;
    const size_t A = (size_t)ch * np + pl;
    lanes[i] = (int)(A & 31);
#pragma unroll
    for (int a = 0; a < 2; a++) {
      if (a >= na) continue;
      // 1/yP is zero exactly for an identity G1 point
      const uint32_t* w = PW + ((((size_t)a * K + k) * 2 + 1) * 12) * np + pl;
      uint32_t nz = 0;
      for (int j = 0; j < 12; j++) nz |= w[(size_t)j * np];
      acta[i][a] = nz != 0;
      size_t bid = ne == 4 ? (A >> 5) * 4 + (size_t)(2 * a + b) : (A >> 5);
      tb[i][a] = ((bid * S + kk) * GS_NUM_LINES) * (size_t)M4_TILE;
      if (acta[i][a]) atomicOr(&masks[bid * S + kk], 1u << lanes[i]);
    }
    act[i] = acta[i][0] || acta[i][1];
    if (act[i]) T.st(i, qx, qy);
    any = any || act[i];
  }
  if (!__syncthreads_or(any)) return;  // block-uniform: the step barriers below need every thread
  int idx = 0;
#pragma unroll 1
  for (int bit = 62; bit >= 0; bit--) {
    const int nl = ((GS_X_ABS >> bit) & 1) ? 2 : 1;
#pragma unroll 1
    for (int w = 0; w < nl; w++, idx++) {
      g2_affine_step<E>(T, Q, act, w == 1, [&](int i, const fp2& lam, const fp2& mu) {
        const int k = kslot[i];
#pragma unroll 1
        for (int a = 0; a < 2; a++) {
          if (!acta[i][a]) continue;
          const uint32_t* pw = PW + ((((size_t)a * K + k) * 2) * 12) * np + pl;
          fp s, wv, v;
#pragma unroll
          for (int j = 0; j < 12; j++) {
            s.l[j] = pw[(size_t)j * np];
            wv.l[j] = pw[(size_t)(12 + j) * np];
          }
          uint32_t* o = tiles + tb[i][a] + (size_t)idx * M4_TILE;
          fp_mul_n(v, mu.c0, wv);
          cq_st_stream(cq_ptr(o, 0, lanes[i]), v);
          fp_mul_n(v, mu.c1, wv);
          cq_st_stream(cq_ptr(o, 1, lanes[i]), v);
          fp_mul_n(v, lam.c0, s);
          cq_st_stream(cq_ptr(o, 2, lanes[i]), v);
          fp_mul_n(v, lam.c1, s);
          cq_st_stream(cq_ptr(o, 3, lanes[i]), v);
        }
      }, [] { __syncthreads(); });
    }
  }
}

// ------------------------------------------------------------------ CRS points: the walk is done once per key
// thread pid (< 6) walks v1.0 v1.1 v2.0 v2.1 W2.0 W2.1 and stores (lambda, mu) of every Miller step
__global__ void k_crs_lines(const crs_dev* __restrict__ crs, fp2* __restrict__ out) {
  const int pid = blockIdx.x * blockDim.x + threadIdx.x;
  if (pid >= 6) return;
  const g2_aff P = pid < 4 ? crs->v[pid >> 1][pid & 1] : crs->w2[pid & 1];
  fp2 Tx[1] = {P.x}, Ty[1] = {P.y}, Qx[1] = {P.x}, Qy[1] = {P.y};
  g2_pts_arr T{Tx, Ty}, Qa{Qx, Qy};
  bool act[1] = {!P.is_inf()};
  int idx = 0;
  for (int bit = 62; bit >= 0; bit--) {
    const int nl = ((GS_X_ABS >> bit) & 1) ? 2 : 1;
    for (int w = 0; w < nl; w++, idx++) {
      fp2 l, m;
      l.set_zero();
      m.set_zero();
      g2_affine_step<1>(T, Qa, act, w == 1, [&](int, const fp2& lam, const fp2& mu) {
        l = lam;
        m = mu;
      }, [] {});
      out[((size_t)pid * GS_NUM_LINES + idx) * 2] = l;
      out[((size_t)pid * GS_NUM_LINES + idx) * 2 + 1] = m;
    }
  }
}
// thread -> (fixed slot f, coordinate b, problem): the tiles of slot fk[f] from the stored (lambda, mu) of CRS point
// fpid[f]*2 + b, evaluated at the two G1 coordinates of the slot: 8 Fp products per step, no walk, no inversion
struct fixed_slots {
  int n;
  int k[4];
  int pid[4];
};
__global__ void __launch_bounds__(128) k_fixed_tiles(const uint32_t* __restrict__ PW, const fp2* __restrict__ lines,
                                                     const crs_dev* __restrict__ crs, uint32_t* __restrict__ tiles,
                                                     uint32_t* __restrict__ masks, size_t p0, size_t np, int K, int S,
                                                     fixed_slots fs) {
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (size_t)fs.n * 2 * np) return;
  (void)p0;
  const size_t pl = q % np;
  const int b = (int)((q / np) & 1), f = (int)(q / (2 * np));
  const int k = fs.k[f], pt = fs.pid[f] * 2 + b;
  const g2_aff P = pt < 4 ? crs->v[pt >> 1][pt & 1] : crs->w2[pt & 1];
  if (P.is_inf()) return;
  const int ch = k / S, kk = k % S;
  const size_t A = (size_t)ch * np + pl;
  const int lane = (int)(A & 31);
#pragma unroll 1
  for (int a = 0; a < 2; a++) {
    const uint32_t* pw = PW + ((((size_t)a * K + k) * 2) * 12) * np + pl;
    fp s, wv;
    uint32_t nz = 0;
#pragma unroll
    for (int j = 0; j < 12; j++) {
      s.l[j] = pw[(size_t)j * np];
      wv.l[j] = pw[(size_t)(12 + j) * np];
      nz |= wv.l[j];
    }
    if (!nz) continue;  // identity G1 point: pair dropped
    const size_t bid = (A >> 5) * 4 + (size_t)(2 * a + b);
    atomicOr(&masks[bid * S + kk], 1u << lane);
    uint32_t* o = tiles + ((bid * S + kk) * GS_NUM_LINES) * (size_t)M4_TILE;
    const fp2* L = lines + (size_t)pt * GS_NUM_LINES * 2;
#pragma unroll 1
    for (int idx = 0; idx < GS_NUM_LINES; idx++, o += M4_TILE) {
      const fp2 lam = L[idx * 2], mu = L[idx * 2 + 1];
      fp v;
      fp_mul_n(v, mu.c0, wv);
      cq_st_stream(cq_ptr(o, 0, lane), v);
      fp_mul_n(v, mu.c1, wv);
      cq_st_stream(cq_ptr(o, 1, lane), v);
      fp_mul_n(v, lam.c0, s);
      cq_st_stream(cq_ptr(o, 2, lane), v);
      fp_mul_n(v, lam.c1, s);
      cq_st_stream(cq_ptr(o, 3, lane), v);
    }
  }
}

// Single-entry products with one accumulator (or acc_stride of them) per proof (gs_verify_each_rand): the first nf slots of
// accumulator A = q * acc_stride pair the proof's folded G1 points with G2 points shared by the whole call (the folded CRS
// elements), whose lines were walked ONCE (gsi::g2_lines).  thread -> (f, q): 32 consecutive proofs of one f per warp, so
// the line loads are uniform and, with acc_stride = 1, the 32 lanes of one tile row are written together.
struct each_pids {
  int n;
  int pid[4];
};
__global__ void __launch_bounds__(128) k_each_fixed_tiles(const uint32_t* __restrict__ PW, const g2_aff* __restrict__ pts,
                                                          const fp2* __restrict__ lines, uint32_t* __restrict__ tiles,
                                                          uint32_t* __restrict__ masks, size_t nq, int acc_stride, int S,
                                                          each_pids ep) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (size_t)ep.n * nq) return;
  const size_t q = id % nq;
  const int f = (int)(id / nq);
  const int pid = ep.pid[f];
  if (pts[pid].is_inf()) return;  // pair dropped
  const size_t A = q * (size_t)acc_stride, k = A * S + f;
  const int lane = (int)(A & 31);
  const uint32_t* pw = PW + k * 2 * 12;  // (nprob = np = 1, one G1 coordinate)
  fp s, wv;
  uint32_t nz = 0;
#pragma unroll
  for (int j = 0; j < 12; j++) {
    s.l[j] = pw[j];
    wv.l[j] = pw[12 + j];
    nz |= wv.l[j];
  }
  if (!nz) return;  // identity G1 point: pair dropped
  const size_t bid = A >> 5;
  atomicOr(&masks[bid * S + f], 1u << lane);
  uint32_t* o = tiles + ((bid * S + f) * GS_NUM_LINES) * (size_t)M4_TILE;
  const fp2* L = lines + (size_t)pid * GS_NUM_LINES * 2;
#pragma unroll 1
  for (int idx = 0; idx < GS_NUM_LINES; idx++, o += M4_TILE) {
    const fp2 lam = L[idx * 2], mu = L[idx * 2 + 1];
    fp v;
    fp_mul_n(v, mu.c0, wv);
    cq_st_stream(cq_ptr(o, 0, lane), v);
    fp_mul_n(v, mu.c1, wv);
    cq_st_stream(cq_ptr(o, 1, lane), v);
    fp_mul_n(v, lam.c0, s);
    cq_st_stream(cq_ptr(o, 2, lane), v);
    fp_mul_n(v, lam.c1, s);
    cq_st_stream(cq_ptr(o, 3, lane), v);
  }
}

// ------------------------------------------------------------------ lone statements: walk ahead, evaluate later
// The walk of a G2 point (lambda, mu per step) does not depend on the G1 side; for a lone statement it is started on
// a second stream while the statement MSM -- which produces some of the G1 slots -- still runs (verify.cu), and the
// lines are evaluated at the G1 points afterwards.  lines[((e*np + pl)*68 + step)*2 + {0,1}], e = walk-list entry.
__global__ void __launch_bounds__(128, 2) k_g2_walk(const g2_aff* __restrict__ Y, fp2* __restrict__ lines, size_t nprob, size_t np,
                                                    int K, const uint32_t* __restrict__ walk, int nwalk) {
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool inrange = q < (size_t)nwalk * np;
  if (!inrange) q = 0;
  const size_t pl = q % np;
  const int e = (int)(q / np);
  const uint32_t we = walk[e];
  const int b = (int)(we >> 31), k = (int)(we & 0x3FFFFFFFu);
  const bool dup = ((we >> 30) & 1) && pl != 0;  // a point shared by all problems is walked for problem 0 only
  const g2_aff P = Y[((size_t)b * K + k) * nprob + pl];
  fp2 Tx[1] = {P.x}, Ty[1] = {P.y}, Qx[1] = {P.x}, Qy[1] = {P.y};
  g2_pts_arr T{Tx, Ty}, Qa{Qx, Qy};
  bool act[1] = {inrange && !dup && !P.is_inf()};
  if (!__syncthreads_or(act[0])) return;
  fp2* out = lines + ((size_t)e * np + pl) * GS_NUM_LINES * 2;
  int idx = 0;
#pragma unroll 1
  for (int bit = 62; bit >= 0; bit--) {
    const int nl = ((GS_X_ABS >> bit) & 1) ? 2 : 1;
#pragma unroll 1
    for (int w = 0; w < nl; w++, idx++) {
      g2_affine_step<1>(T, Qa, act, w == 1, [&](int, const fp2& lam, const fp2& mu) {
        out[idx * 2] = lam;
        out[idx * 2 + 1] = mu;
      }, [] { __syncthreads(); });
    }
  }
}
// ---- the same walk WITHOUT a field inversion per step (lone statements are pure latency: the affine walk above is 68
// dependent steps of ~60 us, two thirds of it the per-step inversion).  The point runs in Jacobian coordinates; with
// x = X / Z^2, y = Y / Z^3 both kinds of step have their slope over the NEW Z coordinate:
//     doubling   lam = 3 x^2 / 2 y = 3 X^2 / (2 Y Z)        = N / Z',   Z' = 2 Y Z         (dbl-2009-l)
//     addition   lam = (y_Q - y_T) / (x_Q - x_T) = r / (Z H) = N / Z',   Z' = Z H           (H = x_Q Z^2 - X, r = y_Q Z^3 - Y)
// so the walk only records (N, X, Y) of the point before the step and Z' (k_g2_walk_jac, one thread per point, ~1 ms),
// and ONE batched inversion of the 68 Z' per point gives every lam and mu = lam x_T - y_T afterwards, all 68 steps in
// parallel (k_g2_lines_from_jac, one block per point).  rec[((e*np + pl)*68 + step)*4 + {0: N, 1: X, 2: Y, 3: Z'}].
__global__ void __launch_bounds__(64) k_g2_walk_jac(const g2_aff* __restrict__ Y, fp2* __restrict__ rec, size_t nprob, size_t np, int K,
                                                    const uint32_t* __restrict__ walk, int nwalk) {
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (size_t)nwalk * np) return;
  const size_t pl = q % np;
  const int e = (int)(q / np);
  const uint32_t we = walk[e];
  const int b = (int)(we >> 31), k = (int)(we & 0x3FFFFFFFu);
  if (((we >> 30) & 1) && pl != 0) return;  // shared by all problems: walked for problem 0 only
  const g2_aff Q = Y[((size_t)b * K + k) * nprob + pl];
  if (Q.is_inf()) return;  // k_eval_tiles drops the pair
  fp2* out = rec + ((size_t)e * np + pl) * GS_NUM_LINES * 4;
  fp2 X = Q.x, Yc = Q.y, Z;
  Z.set_one();
  int idx = 0;
#pragma unroll 1
  for (int bit = 62; bit >= 0; bit--) {
    {  // doubling (a = 0): A = X^2, B = Y^2, C = B^2, D = 2((X+B)^2 - A - C), E = 3A, X3 = E^2 - 2D, Y3 = E(D - X3) - 8C, Z3 = 2YZ
      fp2 A, B, C, D, E, F, t, Z3;
      fp2::sqr(A, X);
      fp2::sqr(B, Yc);
      fp2::sqr(C, B);
      fp2::add(t, X, B);
      fp2::sqr(t, t);
      fp2::sub(t, t, A);
      fp2::sub(t, t, C);
      fp2::dbl(D, t);
      fp2::dbl(E, A);
      fp2::add(E, E, A);
      fp2::mul(t, Yc, Z);
      fp2::dbl(Z3, t);
      out[idx * 4 + 0] = E;
      out[idx * 4 + 1] = X;
      out[idx * 4 + 2] = Yc;
      out[idx * 4 + 3] = Z3;
      fp2::sqr(F, E);
      fp2::sub(t, F, D);
      fp2::sub(X, t, D);
      fp2::sub(t, D, X);
      fp2::mul(t, E, t);
      fp2::dbl(C, C);
      fp2::dbl(C, C);
      fp2::dbl(C, C);
      fp2::sub(Yc, t, C);
      Z = Z3;
      idx++;
    }
    if ((GS_X_ABS >> bit) & 1) {  // T + Q, Q affine
      fp2 Z1Z1, U2, S2, H, r, HH, HHH, V, t, Z3;
      fp2::sqr(Z1Z1, Z);
      fp2::mul(U2, Q.x, Z1Z1);
      fp2::mul(S2, Q.y, Z);
      fp2::mul(S2, S2, Z1Z1);
      fp2::sub(H, U2, X);
      fp2::sub(r, S2, Yc);
      fp2::mul(Z3, Z, H);
      out[idx * 4 + 0] = r;
      out[idx * 4 + 1] = X;
      out[idx * 4 + 2] = Yc;
      out[idx * 4 + 3] = Z3;
      fp2::sqr(HH, H);
      fp2::mul(HHH, H, HH);
      fp2::mul(V, X, HH);
      fp2::sqr(t, r);
      fp2::sub(t, t, HHH);
      fp2::sub(t, t, V);
      fp2 X3;
      fp2::sub(X3, t, V);
      fp2::sub(t, V, X3);
      fp2::mul(t, r, t);
      fp2::mul(HHH, Yc, HHH);
      fp2::sub(Yc, t, HHH);
      X = X3;
      Z = Z3;
      idx++;
    }
  }
}
// block -> walked point (e, pl), thread s < 68 -> Miller step s: lines[((e*np + pl)*68 + s)*2 + {0: lam, 1: mu}]
__global__ void __launch_bounds__(128) k_g2_lines_from_jac(const g2_aff* __restrict__ Y, const fp2* __restrict__ rec, fp2* __restrict__ lines,
                                                           size_t nprob, size_t np, int K, const uint32_t* __restrict__ walk) {
  __shared__ fp sm[2 * 128];
  __shared__ fp2 zinv[GS_NUM_LINES + 1];
  const size_t pt = blockIdx.x;  // e * np + pl
  const size_t pl = pt % np;
  const int e = (int)(pt / np);
  const uint32_t we = walk[e];
  if (((we >> 30) & 1) && pl != 0) return;  // shared by all problems: problem 0's lines serve everyone (block-uniform)
  const g2_aff* Q = &Y[((size_t)(we >> 31) * K + (we & 0x3FFFFFFFu)) * nprob + pl];
  if (Q->x.is_zero() && Q->y.is_zero()) return;  // block-uniform
  const int s = threadIdx.x;
  const fp2* r = rec + (pt * GS_NUM_LINES + (s < GS_NUM_LINES ? s : 0)) * 4;
  fp2 Zn;
  fp nrm;
  nrm.set_zero();
  if (s < GS_NUM_LINES) {
    Zn = r[3];
    fp t;
    fp::sqr(nrm, Zn.c0);
    fp::sqr(t, Zn.c1);
    fp::add(nrm, nrm, t);
  }
  block_batch_inv<128>(nrm, sm);  // 0 (idle threads) passes through
  if (s < GS_NUM_LINES) {         // 1 / Z' = conj(Z') / |Z'|^2
    fp2 zi;
    fp::mul(zi.c0, Zn.c0, nrm);
    fp::mul(zi.c1, Zn.c1, nrm);
    fp::neg(zi.c1, zi.c1);
    zinv[s + 1] = zi;
  }
  if (s == 0) zinv[0].set_one();
  __syncthreads();
  if (s >= GS_NUM_LINES) return;
  fp2 lam, zi = zinv[s], zi2, x, y, mu;
  fp2::mul(lam, r[0], zinv[s + 1]);
  fp2::sqr(zi2, zi);
  fp2::mul(x, r[1], zi2);
  fp2::mul(zi2, zi2, zi);
  fp2::mul(y, r[2], zi2);
  fp2::mul(mu, lam, x);
  fp2::sub(mu, mu, y);
  fp2* o = lines + (pt * GS_NUM_LINES + s) * 2;
  o[0] = lam;
  o[1] = mu;
}

// thread -> (walk entry e, problem): the tiles of slot k, coordinate b from the lines walked ahead
__global__ void __launch_bounds__(128) k_eval_tiles(const uint32_t* __restrict__ PW, const g2_aff* __restrict__ Y,
                                                    const fp2* __restrict__ lines, uint32_t* __restrict__ tiles,
                                                    uint32_t* __restrict__ masks, size_t nprob, size_t np, int K, int S,
                                                    const uint32_t* __restrict__ walk, int nwalk, int ne) {
  size_t q = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= (size_t)nwalk * np) return;
  const size_t pl = q % np;
  const int e = (int)(q / np);
  const uint32_t we = walk[e];
  const int b = (int)(we >> 31), k = (int)(we & 0x3FFFFFFFu);
  const g2_aff* P = &Y[((size_t)b * K + k) * nprob + pl];
  if (P->x.is_zero() && P->y.is_zero()) return;
  const int ch = k / S, kk = k % S;
  const size_t A = (size_t)ch * np + pl;
  const int lane = (int)(A & 31);
  const fp2* L = lines + ((size_t)e * np + (((we >> 30) & 1) ? 0 : pl)) * GS_NUM_LINES * 2;  // (shared point: problem 0's lines)
  const int na = ne == 4 ? 2 : 1;
#pragma unroll 1
  for (int a = 0; a < na; a++) {
    const uint32_t* pw = PW + ((((size_t)a * K + k) * 2) * 12) * np + pl;
    fp s, wv;
    uint32_t nz = 0;
#pragma unroll
    for (int j = 0; j < 12; j++) {
      s.l[j] = pw[(size_t)j * np];
      wv.l[j] = pw[(size_t)(12 + j) * np];
      nz |= wv.l[j];
    }
    if (!nz) continue;  // identity G1 point: pair dropped
    const size_t bid = ne == 4 ? (A >> 5) * 4 + (size_t)(2 * a + b) : (A >> 5);
    atomicOr(&masks[bid * S + kk], 1u << lane);
    uint32_t* o = tiles + ((bid * S + kk) * GS_NUM_LINES) * (size_t)M4_TILE;
#pragma unroll 1
    for (int idx = 0; idx < GS_NUM_LINES; idx++, o += M4_TILE) {
      const fp2 lam = L[idx * 2], mu = L[idx * 2 + 1];
      fp v;
      fp_mul_n(v, mu.c0, wv);
      cq_st_stream(cq_ptr(o, 0, lane), v);
      fp_mul_n(v, mu.c1, wv);
      cq_st_stream(cq_ptr(o, 1, lane), v);
      fp_mul_n(v, lam.c0, s);
      cq_st_stream(cq_ptr(o, 2, lane), v);
      fp_mul_n(v, lam.c1, s);
      cq_st_stream(cq_ptr(o, 3, lane), v);
    }
  }
}

__device__ GS_INL void cp_async16(uint32_t* smem, const uint32_t* g) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(s), "l"(g) : "memory");
}
__device__ GS_INL void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// group (6 warps) = 32 accumulators of entry e (bid = blk*4 + e); warp k = w-power coefficient k (coop12.cuh);
// CQ_GROUPS groups per block.   F[(ch*4 + e) * nprob + p] = conj( prod over the chunk's slots )
__global__ void __launch_bounds__(CQ_BLOCK_THREADS, 1) k_miller4(const uint32_t* __restrict__ tiles,
                                                                const uint32_t* __restrict__ masks, fp12* __restrict__ F,
                                                                size_t nprob, size_t p0, size_t np, int S, int nchunk,
                                                                size_t ngroups, int ne) {
  extern __shared__ __align__(16) uint32_t sm_all[];
  const int grp = threadIdx.x / CQ_GROUP_THREADS, tg = threadIdx.x % CQ_GROUP_THREADS;
  uint32_t* sm = sm_all + (size_t)grp * (M4_SMEM / 4);
  uint32_t* acc = sm;
  uint32_t* tile = sm + 2 * CQ_ACC;
  uint32_t* smask = tile + 2 * M4_TILE;
  uint16_t* slots = (uint16_t*)(smask + M4_MAXS);
  int* nact_s = (int*)(slots + M4_MAXS);
  const int k = tg >> 5, lane = tg & 31;
  // The two groups of a block take ComT entries of EQUAL work: entries (a, 0) carry fewer slots than (a, 1) (the iota_2
  // images have no first coordinate: 8 against 12 pairs per 4x4 PPE proof), and a block that paired entry 0 with entry 1
  // ran its last third with one group = 6 warps.  Block q -> accumulator block q / 2, entries (q & 1) and (q & 1) + 2.
  static_assert(CQ_GROUPS == 2, "entry pairing below assumes two groups per block");
  // (ne = 1, single-entry products: every accumulator block carries the same kind of work, block q -> groups 2q, 2q + 1)
  const size_t bid = ne == 4 ? ((size_t)blockIdx.x >> 1) * 4 + (blockIdx.x & 1) + 2 * (size_t)grp : (size_t)blockIdx.x * 2 + grp;
  if (bid >= ngroups) return;
  if (tg == 0) {
    int n = 0;
    for (int kk = 0; kk < S; kk++) {
      uint32_t m = masks[bid * S + kk];
      if (m) {
        slots[n] = (uint16_t)kk;
        smask[n] = m;
        n++;
      }
    }
    *nact_s = n;
  }
  cq_set_one(k, lane, acc);
  cq_group_sync(grp);
  const int nact = *nact_s;
  int cur = 0;
  if (nact > 0) {
    const int total = GS_NUM_LINES * nact;
    auto issue = [&](int n, int stage) {
      int s = n / nact, i = n - s * nact;
      const uint32_t* src = tiles + ((bid * S + slots[i]) * GS_NUM_LINES + s) * (size_t)M4_TILE;
      uint32_t* dst = tile + stage * M4_TILE;
#pragma unroll
      for (int c = 0; c < M4_TILE / 4 / CQ_GROUP_THREADS; c++) {
        int w = (c * CQ_GROUP_THREADS + tg) * 4;
        cp_async16(dst + w, src + w);
      }
    };
    issue(0, 0);
    cp_async_wait_all();
    cq_group_sync(grp);
    int n = 0;
    for (int bit = 62; bit >= 0; bit--) {
      if (bit != 62) {
        cq_sqr(k, lane, acc + cur * CQ_ACC, acc + (cur ^ 1) * CQ_ACC);
        cq_group_sync(grp);
        cur ^= 1;
      }
      int nl = ((GS_X_ABS >> bit) & 1) ? 2 : 1;
      for (int i = 0; i < nl * nact; i++, n++) {
        if (n + 1 < total) issue(n + 1, (n + 1) & 1);
        int si = i >= nact ? i - nact : i;
        bool active = (smask[si] >> lane) & 1;
        cq_line_mul_u(k, lane, acc + cur * CQ_ACC, acc + (cur ^ 1) * CQ_ACC, tile + (n & 1) * M4_TILE, active);
        cp_async_wait_all();
        cq_group_sync(grp);
        cur ^= 1;
      }
    }
  }
  // conjugate (x < 0) and write out in tower order
  size_t A = (ne == 4 ? (bid >> 2) : bid) * 32 + lane;
  int e = ne == 4 ? (int)(bid & 3) : 0;
  if (A < np * (size_t)nchunk) {
    size_t pl = A % np;
    int ch = (int)(A / np);
    fp2 r;
    cq_ld_coef(r.c0, r.c1, acc + cur * CQ_ACC, k, lane, false, false);
    if (k & 1) fp2::neg(r, r);
    fp2* dst = (fp2*)&F[((size_t)ch * ne + e) * nprob + p0 + pl];
    dst[cq_tower_pos(k)] = r;
  }
}

// ------------------------------------------------------------------ AoS -> slot scatter for ComT ops
// xs[p][k] (Com1), ys[p][k] (Com2) -> X, Y slot arrays
__global__ void k_scatter_pairs(const g1_aff* __restrict__ xs, const g2_aff* __restrict__ ys, g1_aff* __restrict__ X,
                                g2_aff* __restrict__ Y, size_t nprob, int K) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nprob * (size_t)K) return;
  size_t p = id % nprob;
  int k = (int)(id / nprob);
  for (int a = 0; a < 2; a++) {
    X[((size_t)a * K + k) * nprob + p] = xs[(p * K + k) * 2 + a];
    Y[((size_t)a * K + k) * nprob + p] = ys[(p * K + k) * 2 + a];
  }
}

// ------------------------------------------------------------------ small helpers
__global__ void k_fp12_set_one(fp12* out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i].set_one();
}
// out[p*4 + e] = prod_ch F[(ch*4 + e)*nprob + p]   (tower code: a handful of products per problem)
__global__ void k_chunk_product(const fp12* __restrict__ F, fp12* __restrict__ out, size_t nprob, int nchunk, int ne) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nprob * ne) return;
  size_t p = id / ne;
  int e = (int)(id % ne);
  fp12 acc = F[(size_t)e * nprob + p];
  for (int ch = 1; ch < nchunk; ch++) {
    fp12 t = F[((size_t)ch * ne + e) * nprob + p];
    fp12::mul(acc, acc, t);
  }
  out[id] = acc;
}
// iota_T for PPE: (1, 1, 1, t)            data_structures.rs:509-516
__global__ void k_linear_map_ppe(const fp12* t, fp12* out) {
  int e = threadIdx.x;
  if (e >= 4) return;
  if (e == 3)
    out[3] = *t;
  else
    out[e].set_one();
}
// iota_T for the other three types as ONE (Com1, Com2) pair          data_structures.rs:519-540
//   MSMEG1: F(iota_1(t), W2)   MSMEG2: F(W1, iota_2(t))   Quad: F(W1, t W2) = F(t W1, W2)
__global__ void k_linear_map_slots(int type, const void* target, const crs_dev* crs, g1_aff* X, g2_aff* Y) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (type == 1) {
    X[0].set_inf();
    X[1] = *(const g1_aff*)target;
    Y[0] = crs->w2[0];
    Y[1] = crs->w2[1];
  } else if (type == 2) {
    X[0] = crs->w1[0];
    X[1] = crs->w1[1];
    Y[0].set_inf();
    Y[1] = *(const g2_aff*)target;
  } else {
    uint32_t k[8];
    fr_from_mont(k, *(const fr*)target);
    for (int a = 0; a < 2; a++) {
      g1_jac j;
      scalar_mul<FpOps>(j, crs->w1[a], k);
      g1_jac::to_affine(X[a], j);
    }
    Y[0] = crs->w2[0];
    Y[1] = crs->w2[1];
  }
}

}  // namespace gs

int gsi::crs_lines_build(gs_ctx* ctx) {
  if (ctx->crs_lines_valid || !ctx->crs_loaded) return GS_OK;
  if (!ctx->crs_lines) CUDA_TRY(cudaMalloc(&ctx->crs_lines, (size_t)6 * GS_NUM_LINES * 2 * sizeof(fp2)));
  LAUNCH_CFG(k_crs_lines, 6, 32, 0, ctx->crs, ctx->crs_lines);
  ctx->crs_lines_valid = true;
  return GS_OK;
}

int gsi::pairing_init(gs_ctx* ctx) {
  CUDA_TRY(cudaFuncSetAttribute(k_miller4, cudaFuncAttributeMaxDynamicSharedMemorySize, CQ_GROUPS * M4_SMEM));
  return GS_OK;
}

// (coordinate, slot) pairs to walk and the CRS slots with stored lines, from what the shape says about every slot
static void build_walk_list(gs_ctx* ctx, int K, const uint8_t* slot_kind, std::vector<uint32_t>& hwalk, fixed_slots& fs) {
  using namespace gsi;
  fs.n = 0;
  int nfixed = 0;
  for (int k = 0; slot_kind && k < K; k++) nfixed += (slot_kind[k] >= GS_SLOT_FIXED && slot_kind[k] != GS_SLOT_WALK_SHARED) ? 1 : 0;
  const bool use_fixed = ctx->crs_lines_valid && nfixed > 0 && nfixed <= 4;  // no shape has more than 4 CRS slots
  for (int b = 0; b < 2; b++)
    for (int k = 0; k < K; k++) {
      const uint8_t kind = slot_kind ? slot_kind[k] : GS_SLOT_WALK;
      const bool shared = kind == GS_SLOT_WALK_SHARED;
      if (!shared && kind >= GS_SLOT_FIXED && use_fixed) {
        if (b == 0) {
          fs.k[fs.n] = k;
          fs.pid[fs.n] = kind - GS_SLOT_FIXED;
          fs.n++;
        }
        continue;
      }
      if (kind == GS_SLOT_WALK_B1 && b == 0) continue;
      hwalk.push_back(((uint32_t)b << 31) | (shared ? 1u << 30 : 0u) | (uint32_t)k);
    }
}

// Starts the G2 walks of a lone statement on the context's second stream (the Y slots must be complete on the main
// stream); run_pairing_product picks the lines up through `wa`.  No-op (wa->lines = null) outside the latency regime.
int gsi::g2_walk_ahead(gs_ctx* ctx, Scratch& sc, const g2_aff* Y, size_t nprob, int K, const uint8_t* slot_kind, walk_ahead* wa) {
  wa->lines = nullptr;
  std::vector<uint32_t> hwalk;
  fixed_slots fs;
  build_walk_list(ctx, K, slot_kind, hwalk, fs);
  const int nwalk = (int)hwalk.size();
  if (nwalk == 0 || (size_t)((nwalk + 3) / 4) * nprob >= 16384) return GS_OK;
  if (!ctx->stream2) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
  CUDA_TRY(upload(ctx, sc, &wa->dwalk, hwalk.data(), hwalk.size()));
  fp2 *lines, *rec;
  CUDA_TRY(sc.alloc(&lines, (size_t)nwalk * nprob * GS_NUM_LINES * 2));
  CUDA_TRY(sc.alloc(&rec, (size_t)nwalk * nprob * GS_NUM_LINES * 4));
  struct event_guard {  // the fork event is destroyed on every path
    cudaEvent_t e = nullptr;
    ~event_guard() {
      if (e) cudaEventDestroy(e);
    }
  } fork;
  CUDA_TRY(cudaEventCreateWithFlags(&fork.e, cudaEventDisableTiming));
  CUDA_TRY(cudaEventRecord(fork.e, ctx->stream));
  CUDA_TRY(cudaStreamWaitEvent(ctx->stream2, fork.e, 0));
  cudaStream_t main_stream = ctx->stream;
  ctx->stream = ctx->stream2;
  int rc = [&]() -> int {
    // (the inversion-free walk does MORE work per point -- a block per point to turn its 68 records into lines -- and only
    // wins where a point's own dependent chain is the whole cost: a lone statement; 256 statements of a C4 batch walk
    // 50 k points, and there it took 16 ms of the second stream against 8 for the affine walk)
    size_t walked = 0;  // points actually walked: a point shared by all problems counts once
    for (uint32_t we : hwalk) walked += ((we >> 30) & 1) ? 1 : nprob;
    if (ctx->lone_walk_jac && walked <= 4096) {
      LAUNCH_CFG(k_g2_walk_jac, (size_t)nwalk * nprob, 64, 0, Y, rec, nprob, nprob, K, wa->dwalk, nwalk);
      LAUNCH_CFG(k_g2_lines_from_jac, (size_t)nwalk * nprob * 128, 128, 0, Y, rec, lines, nprob, nprob, K, wa->dwalk);
    } else {
      LAUNCH(k_g2_walk, (size_t)nwalk * nprob, Y, lines, nprob, nprob, K, wa->dwalk, nwalk);
    }
    return GS_OK;
  }();
  ctx->stream = main_stream;
  // whatever happened to the launch, the main stream must not free `lines` / `dwalk` before stream2 is past this point
  wa->ctx = ctx;
  if (cudaEventCreateWithFlags(&wa->done, cudaEventDisableTiming) != cudaSuccess || cudaEventRecord(wa->done, ctx->stream2) != cudaSuccess) {
    cudaStreamSynchronize(ctx->stream2);
    if (wa->done) cudaEventDestroy(wa->done);
    wa->done = nullptr;
    if (rc) return rc;
    FAIL(GS_ECUDA, "walk-ahead: event creation failed");
  }
  if (rc) return rc;
  wa->lines = lines;
  wa->nwalk = nwalk;
  return GS_OK;
}

// the inversion-free walk of k_g2_walk_jac / k_g2_lines_from_jac over n points (one "problem", slot k = point k)
int gsi::g2_lines(gs_ctx* ctx, Scratch& sc, const g2_aff* pts, int n, fp2** lines) {
  std::vector<uint32_t> hwalk(n);
  for (int i = 0; i < n; i++) hwalk[i] = (uint32_t)i;
  uint32_t* dwalk;
  fp2* rec;
  CUDA_TRY(upload(ctx, sc, &dwalk, hwalk.data(), hwalk.size()));
  CUDA_TRY(sc.alloc(lines, (size_t)n * GS_NUM_LINES * 2));
  CUDA_TRY(sc.alloc(&rec, (size_t)n * GS_NUM_LINES * 4));
  LAUNCH_CFG(k_g2_walk_jac, (size_t)n, 64, 0, pts, rec, (size_t)1, (size_t)1, n, dwalk, n);
  LAUNCH_CFG(k_g2_lines_from_jac, (size_t)n * 128, 128, 0, pts, rec, *lines, (size_t)1, (size_t)1, n, dwalk);
  return GS_OK;
}

// ------------------------------------------------------------------ pairing-product pipeline
// X, Y: device slot arrays [2][K][nprob].  Produces either ComT values (out_comt, AoS [p][4]) or
// per-entry verdict bytes ok4[4][nprob] (compared with 1 / target).
// Problems are processed in passes of `pc` so that the evaluated-line tiles stay within ctx->tile_budget
// bytes of HBM; a pass is sized to a whole number of k_miller4 waves (2 groups x 148 SMs x 32 accumulators
// / 4 entries = 2,368 problems per wave) when the batch is large enough.
// ne = 1 (gs_verify_batch_rand): SINGLE-entry products prod_k e(X_k, Y_k) over arrays X[K][nprob], Y[K][nprob]; every
// accumulator takes exactly S = S_force slots (K a multiple of it, S a multiple of 4), un-exponentiated result in out_partial,
// or, with `each` (gs_verify_each_rand), one un-exponentiated result per accumulator in each->F.
int gsi::run_pairing_product(gs_ctx* ctx, Scratch& sc, const g1_aff* X, const g2_aff* Y, size_t nprob, int K,
                               fp12* out_comt, uint8_t* ok4, const fp12* target, fp12* out_partial, const uint8_t* slot_kind,
                               const walk_ahead* wa, int ne, int S_force, const acc_each* each) {
  if (ne != 4 && (ne != 1 || nprob != 1 || (!out_partial == !each) || slot_kind || wa || S_force < 4 || S_force % 4 || K % S_force))
    FAIL(GS_EARG, "pairing product: bad single-entry configuration");
  if (each && (ne != 1 || each->nf < 0 || each->nf > 4 || each->nf > S_force || each->acc_stride < 1 || (K / S_force) % each->acc_stride))
    FAIL(GS_EARG, "pairing product: bad per-accumulator configuration");
  const int na = ne == 4 ? 2 : 1;
  const size_t wave = 2368;
  if (K == 0) {  // a shard that owns no slot: empty product
    if (!out_partial) FAIL(GS_EARG, "pairing product over zero slots");
    LAUNCH(k_fp12_set_one, nprob * ne, out_partial, nprob * ne);
    return GS_OK;
  }
  // split the slots of a big statement over several accumulators when there are few problems
  int S = K, nchunk = 1;
  if (nprob < wave && K > 2) {
    size_t c = (wave + nprob - 1) / nprob;
    // at least 2 slots per chunk -- unless one slot per accumulator still fits a single wave: then the Miller chain
    // of a lone statement is 62 squarings + 68 line steps instead of 62 + 136 (latency form)
    const size_t cmax = nprob * (size_t)K <= wave ? (size_t)K : (size_t)(K + 1) / 2;
    if (c > cmax) c = cmax;
    if (c < 1) c = 1;
    S = (int)((K + c - 1) / c);
  }
  if (S > M4_MAXS) S = M4_MAXS;
  if (ne == 1) S = S_force;
  nchunk = (K + S - 1) / S;
  const size_t per_prob = (size_t)ne * nchunk * S * GS_NUM_LINES * M4_TILE * 4 / 32;  // tile bytes per problem
  if (ne == 1 && per_prob > ctx->tile_budget) FAIL(GS_EDIM, "pairing product: single-entry pass exceeds the tile budget");
  size_t pc = ctx->tile_budget / per_prob;
  if (pc >= nprob) {
    pc = nprob;
  } else {
    if (pc > wave) pc -= pc % wave;
    if (pc < 32) pc = 32;
    pc -= pc % 32;
  }
  const size_t nblk_max = ((pc * nchunk + 31) / 32) * ne;
  // which (coordinate, slot) pairs have a point to walk; which slots are CRS points with stored lines
  std::vector<uint32_t> hwalk;
  fixed_slots fs;
  if (ne == 4) {
    build_walk_list(ctx, K, slot_kind, hwalk, fs);
  } else {
    // thread g of the walk kernel takes the entries 4g .. 4g+3: slot quad r of accumulator ch, with g = r * nchunk + ch, so
    // that the 32 threads of a warp write the 32 lanes of ONE tile (consecutive accumulators, same slot) in 512-B rows
    fs.n = 0;
    hwalk.resize((size_t)K);
    for (int r = 0; r < S / 4; r++)
      for (int ch = 0; ch < nchunk; ch++)
        for (int i = 0; i < 4; i++) hwalk[4 * ((size_t)r * nchunk + ch) + i] = (uint32_t)(ch * S + 4 * r + i);
  }
  const int nwalk = (int)hwalk.size();
  if (wa && (!wa->lines || wa->nwalk != nwalk || pc < nprob)) wa = nullptr;  // lines walked ahead only for a single pass
  uint32_t* dwalk;
  if (wa)
    dwalk = wa->dwalk;
  else
    CUDA_TRY(upload(ctx, sc, &dwalk, hwalk.data(), hwalk.size()));
  uint32_t *tiles, *masks, *PW;
  fp12* F;
  CUDA_TRY(sc.alloc(&PW, (size_t)na * K * 24 * pc));
  CUDA_TRY(sc.alloc(&tiles, nblk_max * S * GS_NUM_LINES * (size_t)M4_TILE));
  CUDA_TRY(sc.alloc(&masks, nblk_max * S));
  if (each)
    F = each->F;
  else
    CUDA_TRY(sc.alloc(&F, (size_t)nchunk * ne * nprob));
  for (size_t p0 = 0; p0 < nprob; p0 += pc) {
    size_t np = nprob - p0 < pc ? nprob - p0 : pc;
    size_t nblk = ((np * nchunk + 31) / 32) * ne;
    CUDA_TRY(cudaMemsetAsync(masks, 0, nblk * S * sizeof(uint32_t), ctx->stream));
    LAUNCH(k_g1_prep, (size_t)na * K * np, X, PW, nprob, p0, np, K, na);
    // (6 points per thread was measured too: 162.6 ms vs 151.0 ms per 65,536 proofs -- the extra local memory costs
    // more than the shared inversion saves)
    if (fs.n) LAUNCH(k_fixed_tiles, (size_t)fs.n * 2 * np, PW, ctx->crs_lines, ctx->crs, tiles, masks, p0, np, K, S, fs);
    if (each && each->nf) {
      each_pids ep;
      ep.n = each->nf;
      for (int f = 0; f < 4; f++) ep.pid[f] = each->pid[f];
      const size_t nq = (size_t)nchunk / each->acc_stride;
      LAUNCH(k_each_fixed_tiles, (size_t)ep.n * nq, PW, each->pts, each->lines, tiles, masks, nq, each->acc_stride, S, ep);
    }
    if (wa) {
      CUDA_TRY(cudaStreamWaitEvent(ctx->stream, wa->done, 0));
      LAUNCH(k_eval_tiles, (size_t)nwalk * np, PW, Y, wa->lines, tiles, masks, nprob, np, K, S, dwalk, nwalk, ne);
    } else if ((size_t)((nwalk + 3) / 4) * np < 16384 && ctx->lone_walk_jac && p0 == 0 && np == nprob && (size_t)nwalk * np <= 4096) {
      // few points (a lone pairing / ComT product / CRS generation): the inversion-free walk, then the evaluation
      fp2 *lines, *rec;
      CUDA_TRY(sc.alloc(&lines, (size_t)nwalk * np * GS_NUM_LINES * 2));
      CUDA_TRY(sc.alloc(&rec, (size_t)nwalk * np * GS_NUM_LINES * 4));
      LAUNCH_CFG(k_g2_walk_jac, (size_t)nwalk * np, 64, 0, Y, rec, nprob, np, K, dwalk, nwalk);
      LAUNCH_CFG(k_g2_lines_from_jac, (size_t)nwalk * np * 128, 128, 0, Y, rec, lines, nprob, np, K, dwalk);
      LAUNCH(k_eval_tiles, (size_t)nwalk * np, PW, Y, lines, tiles, masks, nprob, np, K, S, dwalk, nwalk, ne);
    } else if ((size_t)((nwalk + 3) / 4) * np < 16384 && ne == 4)
      LAUNCH_CFG((k_g2_prepare4<1, 2>), (size_t)nwalk * np, 128, 0, PW, Y, tiles, masks, nprob, p0, np, K, S, dwalk, nwalk, ne);
    else if (ctx->prep_variant == 4)
      LAUNCH_CFG((k_g2_prepare4<4, 4>), (size_t)((nwalk + 3) / 4) * np, 128, 0, PW, Y, tiles, masks, nprob, p0, np, K, S, dwalk, nwalk, ne);
    else
      LAUNCH_CFG((k_g2_prepare4<4, 5>), (size_t)((nwalk + 3) / 4) * np, 128, 0, PW, Y, tiles, masks, nprob, p0, np, K, S, dwalk, nwalk, ne);
    LAUNCH_CFG(k_miller4, ((nblk + CQ_GROUPS - 1) / CQ_GROUPS) * CQ_BLOCK_THREADS, CQ_BLOCK_THREADS, CQ_GROUPS * M4_SMEM, tiles, masks,
               F, nprob, p0, np, S, nchunk, nblk, ne);
  }
  if (each) return GS_OK;
  const fp12* Fr = F;
  if (out_partial) {  // sharded statement: hand back the un-exponentiated Miller products, one per ComT entry
    int rc = gsi::reduce_chunks(ctx, sc, &Fr, nprob, &nchunk, 1, ne);
    if (rc) return rc;
    LAUNCH(k_chunk_product, nprob * ne, Fr, out_partial, nprob, nchunk, ne);
    return GS_OK;
  }
  if (nchunk > 12) {
    int rc = gsi::reduce_chunks(ctx, sc, &Fr, nprob, &nchunk, 12);
    if (rc) return rc;
  }
  return gsi::launch_final_exp(ctx, Fr, nprob, nchunk, out_comt, ok4, target);
}

static int comt_pairing_impl(gs_ctx* ctx, size_t nprob, int K, const gs_com1* xs, const gs_com2* ys, gs_comt* out) {
  if (!ctx || !xs || !ys || !out) return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  g1_aff *dx, *X;
  g2_aff *dy, *Y;
  fp12* dout;
  size_t np = nprob * K;
  CUDA_TRY(upload(ctx, sc, &dx, xs, np * 2));
  CUDA_TRY(upload(ctx, sc, &dy, ys, np * 2));
  CUDA_TRY(sc.alloc(&X, np * 2));
  CUDA_TRY(sc.alloc(&Y, np * 2));
  CUDA_TRY(sc.alloc(&dout, nprob * 4));
  LAUNCH(k_scatter_pairs, np, dx, dy, X, Y, nprob, K);
  int rc = gsi::run_pairing_product(ctx, sc, X, Y, nprob, K, dout, nullptr, nullptr, nullptr);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(out, dout, nprob * 4 * sizeof(fp12), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}


extern "C" {

int gs_comt_pairing(gs_ctx* ctx, size_t count, const gs_com1* xs, const gs_com2* ys, gs_comt* out) {
  if (!ctx) return GS_EARG;
  if (count == 0) return GS_OK;
  return comt_pairing_impl(ctx, count, 1, xs, ys, out);
}

int gs_comt_pairing_sum(gs_ctx* ctx, size_t k, const gs_com1* xs, const gs_com2* ys, gs_comt* out) {
  if (!ctx || !out) return GS_EARG;
  if (k == 0) {  // empty sum = ComT::zero() = four GT identities
    CUDA_TRY(cudaSetDevice(ctx->device));
    Scratch sc(ctx);
    fp12* d;
    CUDA_TRY(sc.alloc(&d, 4));
    LAUNCH(k_fp12_set_one, 4, d, (size_t)4);
    CUDA_TRY(cudaMemcpyAsync(out, d, 4 * sizeof(fp12), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return GS_OK;
  }
  if (k > (size_t)1 << 24) FAIL(GS_EDIM, "pairing_sum: too many pairs");
  return comt_pairing_impl(ctx, 1, (int)k, xs, ys, out);
}

int gs_pairing(gs_ctx* ctx, size_t count, const gs_g1* ps, const gs_g2* qs, gs_gt* out) {
  if (!ctx || !ps || !qs || !out) return GS_EARG;
  if (count == 0) return GS_OK;
  // e(P,Q) = entry (0,0) of F((P,O),(Q,O))
  std::vector<gs_com1> xs(count);
  std::vector<gs_com2> ys(count);
  std::vector<gs_comt> res(count);
  memset(xs.data(), 0, count * sizeof(gs_com1));
  memset(ys.data(), 0, count * sizeof(gs_com2));
  for (size_t i = 0; i < count; i++) {
    xs[i].p[0] = ps[i];
    ys[i].p[0] = qs[i];
  }
  int rc = comt_pairing_impl(ctx, count, 1, xs.data(), ys.data(), res.data());
  if (rc) return rc;
  for (size_t i = 0; i < count; i++) out[i] = res[i].e[0];
  return GS_OK;
}

int gs_comt_linear_map(gs_ctx* ctx, int type, const void* target, gs_comt* out) {
  if (!ctx || !target || !out) return GS_EARG;
  if (type < 0 || type > 3) FAIL(GS_EARG, "linear_map: bad equation type");
  if (type != GS_PPE && !ctx->crs_loaded) FAIL(GS_EARG, "linear_map: no CRS loaded");
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  g1_aff* X;
  g2_aff* Y;
  fp12* dout;
  void* dt;
  size_t tsz = type == GS_PPE ? sizeof(fp12) : type == GS_MSMEG1 ? sizeof(g1_aff) : type == GS_MSMEG2 ? sizeof(g2_aff) : sizeof(fr);
  CUDA_TRY(upload(ctx, sc, (uint8_t**)&dt, target, tsz));
  CUDA_TRY(sc.alloc(&X, 2));
  CUDA_TRY(sc.alloc(&Y, 2));
  CUDA_TRY(sc.alloc(&dout, 4));
  if (type == GS_PPE) {
    LAUNCH(k_linear_map_ppe, 4, (const fp12*)dt, dout);
  } else {
    LAUNCH(k_linear_map_slots, 1, type, dt, ctx->crs, X, Y);
    int rc = gsi::run_pairing_product(ctx, sc, X, Y, 1, 1, dout, nullptr, nullptr, nullptr);
    if (rc) return rc;
  }
  CUDA_TRY(cudaMemcpyAsync(out, dout, 4 * sizeof(fp12), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}


}  // extern "C"
