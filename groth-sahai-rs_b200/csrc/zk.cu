// Zero knowledge for PPE targets given as pairs (Groth & Sahai, EUROCRYPT 2008, PAPERS.md; not in the reference).  The
// simulator absorbs a PPE target only when it is 1, so a PPE
//     sum_j e(A_j, Y_j) + sum_i e(X_i, B_i) + sum_ij gamma_ij e(X_i, Y_j) = sum_k e(P_k, Q_k)
// is proved as an augmented statement: one PPE' with target 1 over the x-variables (X | Z), constants b' = (B | -Q) and
// Gamma with K zero rows, and K MSMEG1 equations L_k : Z_k - delta P_k = O (a = [-P_k], b = [1], Gamma = [[0]]) whose
// scalar y-variable delta has the FIXED commitment W2 = 1 W2 + 0 v[0], rebuilt by the verifier from its CRS.  Under a
// binding CRS W2 binds delta = 1, so Z_k = P_k and PPE' is the original equation; under a hiding CRS W2 = t2 v[0] is also
// the commitment of delta = 0 with randomness t2, which is how the simulator proves L_k with Z_k = O.
// The drivers below own this layout and run the existing impls on it: commit + prove, simulate, rerandomise, verify, and the
// randomised per-statement check of verify.cu (gsi::zk_each_rand_dev).  Arrays are host arrays in the engine's proof-major
// layout; the only kernel of its own is the AND of the 1 + K verdicts (the fixed-base sums of rerandomised L_k are
// k_fixed_com_add of prover_impl.cuh).
#include <algorithm>
#include <cstddef>

#include "ctx.h"

using namespace gs;
using namespace gsi;

namespace {

// out[i] = ok_ppe[i] & ok_lin[i][0] & ... & ok_lin[i][K - 1]
__global__ void k_zk_and(const uint8_t* __restrict__ ok_ppe, const uint8_t* __restrict__ ok_lin, size_t count, int K,
                         uint8_t* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  uint8_t ok = ok_ppe[i];
  for (int k = 0; k < K; k++) ok &= ok_lin[i * K + k];
  out[i] = ok;
}

template <class F, class P>
P negated(const P& p) {  // -p (the identity, all-zero bytes, stays itself)
  P r = p;
  F::neg(reinterpret_cast<Aff<F>&>(r).y, reinterpret_cast<Aff<F>&>(r).y);
  return r;
}

// The statement arrays of the augmented statement of `count` PPEs with K target pairs each (host, proof-major)
struct zk_layout {
  std::vector<gs_g2> b;          // PPE': [count][m + K]     = B | -Q
  std::vector<gs_fr> gamma;      // PPE': [count][m + K][n]  = Gamma, then K zero rows
  std::vector<gs_gt> ones;       // PPE': [count]            target 1
  std::vector<gs_g1> lin_a;      // L_k : [count][K]         -P_k (left empty without tp: rerandomisation never reads it)
  std::vector<gs_fr> lin_b;      // L_k : [count][K]         1 (b, and delta of the real prover)
  std::vector<gs_fr> lin_gamma;  // L_k : [count][K]         0
  zk_layout(size_t count, size_t m, size_t n, size_t K, const gs_g2* b_consts, const gs_fr* gm, const gs_g1* tp, const gs_g2* tq)
      : b(count * (m + K)), gamma(count * (m + K) * n), ones(count), lin_a(tp ? count * K : 0), lin_b(count * K),
        lin_gamma(count * K) {
    fp12 one12;
    one12.set_one();
    fr one;
    for (int i = 0; i < 8; i++) one.l[i] = FR_ONE_MONT(i);
    for (size_t i = 0; i < count; i++) {
      memcpy(&b[i * (m + K)], b_consts + i * m, m * sizeof(gs_g2));
      memcpy(&gamma[i * (m + K) * n], gm + i * m * n, m * n * sizeof(gs_fr));
      memcpy(&ones[i], &one12, sizeof(gs_gt));
      for (size_t k = 0; k < K; k++) {
        b[i * (m + K) + m + k] = negated<Fp2Ops>(tq[i * K + k]);
        if (tp) lin_a[i * K + k] = negated<FpOps>(tp[i * K + k]);
        memcpy(&lin_b[i * K + k], &one, sizeof(gs_fr));
      }
    }
  }
};

// rows m .. m + K - 1 of every statement's R (x_rand[count][m + K][2]): the randomness of Z_1 .. Z_K, [count][K][2]
std::vector<gs_fr> z_rand(const gs_fr* x_rand, size_t count, size_t m, size_t K) {
  std::vector<gs_fr> r(count * K * 2);
  for (size_t i = 0; i < count; i++) memcpy(&r[i * K * 2], x_rand + (i * (m + K) + m) * 2, K * 2 * sizeof(gs_fr));
  return r;
}

// argument checks shared by the three entry points, in gs_simulate_batch's order; count == 0 passes (GS_OK)
int zk_args(gs_ctx* ctx, const char* what, size_t count, size_t m, size_t n, size_t K, bool set) {
  if (!ctx) return GS_EARG;
  if (!ctx->crs_loaded) FAIL(GS_EARG, std::string(what) + ": no CRS loaded");
  if (count == 0) return GS_OK;
  if (m == 0 || n == 0) FAIL(GS_EDIM, std::string(what) + ": empty variable list");
  if (K == 0) FAIL(GS_EDIM, std::string(what) + ": no target pair (a target-1 PPE needs no augmented statement)");
  if (m > 1 << 20 || n > 1 << 20 || K > 1 << 20 || m + K > 1 << 20) FAIL(GS_EDIM, std::string(what) + ": too many variables");
  return set ? GS_OK : GS_EARG;
}


// the host arrays of a verify call (proof-major)
struct zk_host {
  size_t m, n, K;
  const gs_g1* a_consts;
  const gs_com1* xcoms;
  const gs_com2* ycoms;
  const gs_com2* pi;
  const gs_com1* theta;
  const gs_com2* lin_pi;
  const gs_com1* lin_theta;
};

// delta's commitment is never taken from the proof: W2 of the loaded CRS, once per call
int crs_w2(gs_ctx* ctx, gs_com2* w2) {
  CUDA_TRY(cudaMemcpyAsync(w2, &ctx->crs->w2[0], sizeof(*w2), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

// statements per upload: at most 4 verify passes of L_k, so that device scratch does not grow with the batch (C5 at
// K = 1, 65,536 statements, is one chunk; within a chunk verify_impl alternates its passes between two streams)
size_t zk_chunk(const gs_ctx* ctx, size_t K) { return std::max<size_t>(1, 4 * ctx->verify_batch_max / K); }

// device copies of statements [off, off + cn) in the augmented layout, PPE''s target left out: PPE' (A, B, G, c, d, pi, th)
// and the cn * K equations L_k (La, Lb, Lg, Lt = O, Lc, Ld = W2, Lpi, Lth)
struct zk_dev {
  g1_aff *A, *La, *Lt;
  g2_aff *B, *Ld;
  fr *G, *Lb, *Lg;
  gs_com1 *c, *th, *Lc, *Lth;
  gs_com2 *d, *pi, *Lpi;
};
int zk_upload(gs_ctx* ctx, Scratch& sc, const zk_host& h, const zk_layout& L, const gs_com2& w2, size_t off, size_t cn, zk_dev* d) {
  const size_t m = h.m, n = h.n, K = h.K, mk = m + K, nl = cn * K;
  const std::vector<gs_com2> lin_d(nl, w2);
  const std::vector<gs_g1> origin(nl);
  CUDA_TRY(upload(ctx, sc, &d->A, h.a_consts + off * n, cn * n));
  CUDA_TRY(upload(ctx, sc, &d->B, L.b.data(), cn * mk));
  CUDA_TRY(upload(ctx, sc, &d->G, L.gamma.data(), cn * mk * n));
  CUDA_TRY(upload(ctx, sc, &d->c, h.xcoms + off * mk, cn * mk));
  CUDA_TRY(upload(ctx, sc, &d->d, h.ycoms + off * n, cn * n));
  CUDA_TRY(upload(ctx, sc, &d->pi, h.pi + off * 2, cn * 2));
  CUDA_TRY(upload(ctx, sc, &d->th, h.theta + off * 2, cn * 2));
  CUDA_TRY(upload(ctx, sc, &d->La, L.lin_a.data(), nl));
  CUDA_TRY(upload(ctx, sc, &d->Lb, L.lin_b.data(), nl));
  CUDA_TRY(upload(ctx, sc, &d->Lg, L.lin_gamma.data(), nl));
  CUDA_TRY(upload(ctx, sc, &d->Lt, origin.data(), nl));
  CUDA_TRY(upload(ctx, sc, &d->Ld, lin_d.data(), 2 * nl));
  CUDA_TRY(upload(ctx, sc, &d->Lpi, h.lin_pi + off * K * 2, nl * 2));
  CUDA_TRY(upload(ctx, sc, &d->Lth, h.lin_theta + off * K, nl));
  // L_k's x-commitment is c_{m+k} of PPE': the last K commitments of every statement
  CUDA_TRY(sc.alloc(&d->Lc, nl));
  CUDA_TRY(cudaMemcpy2DAsync(d->Lc, K * sizeof(gs_com1), d->c + m, mk * sizeof(gs_com1), K * sizeof(gs_com1), cn,
                             cudaMemcpyDeviceToDevice, ctx->stream));
  return GS_OK;
}

// The nl = count * K equations L_k of a rerandomised proof under R'_{m+k} (zr, [nl][2]) and T'_k (lin_rand, [nl][1][2]),
// delta's fresh randomness 0.  With Gamma = 0 and b = [1], gs_rerandomize's formula leaves fixed-base terms only:
//   lin_pi'_c = lin_pi_c + R'[m+k][c] W2 - T'_k[c] v[0]   (c = 0, 1)        lin_theta' = lin_theta + T'_k[0] u[0] + T'_k[1] u[1]
// c_{m+k} is rerandomised with PPE'; W2 is neither recomputed nor output, and P_k is never read (its terms carry delta's 0).
int lin_rerandomize(gs_ctx* ctx, size_t nl, const std::vector<gs_fr>& zr, const gs_fr* lin_rand, const gs_com2* lin_pi,
                    const gs_com1* lin_theta, gs_com2* out_lin_pi, gs_com1* out_lin_theta) {
  std::vector<gs_fr> neg_t(nl * 2);  // -T'_k[c] (r - x on the limbs; 0 stays 0)
  for (size_t j = 0; j < nl * 2; j++) fr::neg(reinterpret_cast<fr&>(neg_t[j]), reinterpret_cast<const fr&>(lin_rand[j]));
  Scratch sc(ctx);
  fr *dz, *dnt, *dt;
  g2_aff *dpi, *dpo;
  g1_aff *dth, *dto;
  CUDA_TRY(upload(ctx, sc, &dz, zr.data(), nl * 2));
  CUDA_TRY(upload(ctx, sc, &dnt, neg_t.data(), nl * 2));
  CUDA_TRY(upload(ctx, sc, &dt, lin_rand, nl * 2));
  CUDA_TRY(upload(ctx, sc, &dpi, lin_pi, nl * 2 * 2));
  CUDA_TRY(upload(ctx, sc, &dth, lin_theta, nl * 2));
  CUDA_TRY(sc.alloc(&dpo, nl * 2 * 2));
  CUDA_TRY(sc.alloc(&dto, nl * 2));
  // pi: 2 nl Com2 (c = 0, 1 of every L_k) with bases W2 (2) and v[0] (0); theta: nl Com1 with bases u[0] (0), u[1] (1)
  if (int rc = fixed_com_add<Fp2Ops>(ctx, nl * 2, 2, 0, dz, 1, dnt, 1, dpi, dpo)) return rc;
  if (int rc = fixed_com_add<FpOps>(ctx, nl, 0, 1, dt, 2, dt + 1, 2, dth, dto)) return rc;
  CUDA_TRY(cudaMemcpyAsync(out_lin_pi, dpo, nl * 2 * sizeof(gs_com2), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(out_lin_theta, dto, nl * sizeof(gs_com1), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}
}  // namespace

extern "C" {

int gs_zk_ppe_prove_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts, const gs_g2* b_consts,
                          const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq, const gs_g1* xvars, const gs_g2* yvars,
                          const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, const gs_fr* lin_rand,
                          gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta, gs_com2* out_lin_pi,
                          gs_com1* out_lin_theta) {
  const bool set = a_consts && b_consts && gamma && tp && tq && xvars && yvars && x_rand && y_rand && pf_rand && lin_rand &&
                   out_xcoms && out_ycoms && out_pi && out_theta && out_lin_pi && out_lin_theta;
  if (int rc = zk_args(ctx, "zk_ppe_prove", count, m, n, K, set)) return rc;
  if (count == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const zk_layout L(count, m, n, K, b_consts, gamma, tp, tq);
  const size_t mk = m + K;
  std::vector<gs_g1> xz(count * mk);  // the x-variables of PPE': X | Z with Z = P
  for (size_t i = 0; i < count; i++) {
    memcpy(&xz[i * mk], xvars + i * m, m * sizeof(gs_g1));
    memcpy(&xz[i * mk + m], tp + i * K, K * sizeof(gs_g1));
  }
  // the commitments as gs_batch_commit_g1 / _g2: c = iota_1(X | P) + R u, d = iota_2(Y) + S v
  int rc = batch_commit_impl<FpOps>(ctx, count * mk, 0, 1, x_rand, 2, x_rand + 1, 2, 2 * count * mk, xz.data(), out_xcoms);
  if (rc) return rc;
  if ((rc = batch_commit_impl<Fp2Ops>(ctx, count * n, 0, 1, y_rand, 2, y_rand + 1, 2, 2 * count * n, yvars, out_ycoms))) return rc;
  if ((rc = prove_impl(ctx, GS_PPE, count, mk, n, a_consts, L.b.data(), L.gamma.data(), xz.data(), yvars, x_rand, y_rand, pf_rand,
                       false, out_pi, out_theta)))
    return rc;
  // L_k with Z_k = P_k under row m + k of R, delta = 1 under randomness 0 (its commitment is W2)
  const std::vector<gs_fr> zr = z_rand(x_rand, count, m, K), zero(count * K);
  return prove_impl(ctx, GS_MSMEG1, count * K, 1, 1, L.lin_a.data(), L.lin_b.data(), L.lin_gamma.data(), tp, L.lin_b.data(), zr.data(),
                    zero.data(), lin_rand, false, out_lin_pi, out_lin_theta);
}

int gs_zk_ppe_simulate_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts, const gs_g2* b_consts,
                             const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq, const gs_fr* x_rand, const gs_fr* y_rand,
                             const gs_fr* pf_rand, const gs_fr* lin_rand, const gs_fr* tkey, gs_com1* out_xcoms, gs_com2* out_ycoms,
                             gs_com2* out_pi, gs_com1* out_theta, gs_com2* out_lin_pi, gs_com1* out_lin_theta) {
  const bool set = a_consts && b_consts && gamma && tp && tq && x_rand && y_rand && pf_rand && lin_rand && tkey && out_xcoms &&
                   out_ycoms && out_pi && out_theta && out_lin_pi && out_lin_theta;
  if (int rc = zk_args(ctx, "zk_ppe_simulate", count, m, n, K, set)) return rc;
  if (count == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  if (int rc = sim_key_check(ctx, tkey)) return rc;  // before anything is written
  const zk_layout L(count, m, n, K, b_consts, gamma, tp, tq);
  const size_t mk = m + K;
  // PPE' has target 1: commitments of O under R, S (Z = O included), the proof with every witness O
  int rc = simulate_impl(ctx, GS_PPE, count, mk, n, a_consts, L.b.data(), L.gamma.data(), L.ones.data(), x_rand, y_rand, pf_rand,
                         false, tkey, out_xcoms, out_ycoms, out_pi, out_theta);
  if (rc) return rc;
  // L_k with Z_k = O under row m + k of R and delta = 0 under randomness t2 (whose commitment is W2 too): the MSMEG1
  // simulator with target O, without its commitments (c_{m+k} is written above, W2 is not part of the proof)
  const std::vector<gs_fr> zr = z_rand(x_rand, count, m, K), t2(count * K, tkey[1]);
  const std::vector<gs_g1> origin(count * K);
  return simulate_impl(ctx, GS_MSMEG1, count * K, 1, 1, L.lin_a.data(), L.lin_b.data(), L.lin_gamma.data(), origin.data(), zr.data(),
                       t2.data(), lin_rand, false, tkey, nullptr, nullptr, out_lin_pi, out_lin_theta, false);
}

int gs_zk_ppe_rerandomize_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                                const gs_g2* b_consts, const gs_fr* gamma, const gs_g2* tq, const gs_com1* xcoms,
                                const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const gs_com2* lin_pi,
                                const gs_com1* lin_theta, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand,
                                const gs_fr* lin_rand, gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta,
                                gs_com2* out_lin_pi, gs_com1* out_lin_theta) {
  const bool set = a_consts && b_consts && gamma && tq && xcoms && ycoms && pi && theta && lin_pi && lin_theta && x_rand && y_rand &&
                   pf_rand && lin_rand && out_xcoms && out_ycoms && out_pi && out_theta && out_lin_pi && out_lin_theta;
  if (int rc = zk_args(ctx, "zk_ppe_rerandomize", count, m, n, K, set)) return rc;
  if (count == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const zk_layout L(count, m, n, K, b_consts, gamma, nullptr, tq);
  // PPE': gs_rerandomize_batch of the augmented statement under R', S', T' -- c_{m+k} included
  int rc = rerandomize_impl(ctx, GS_PPE, count, m + K, n, a_consts, L.b.data(), L.gamma.data(), xcoms, ycoms, pi, theta, x_rand,
                            y_rand, pf_rand, false, out_xcoms, out_ycoms, out_pi, out_theta);
  if (rc) return rc;
  return lin_rerandomize(ctx, count * K, z_rand(x_rand, count, m, K), lin_rand, lin_pi, lin_theta, out_lin_pi, out_lin_theta);
}

int gs_zk_ppe_verify_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts, const gs_g2* b_consts,
                           const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq, const gs_com1* xcoms, const gs_com2* ycoms,
                           const gs_com2* pi, const gs_com1* theta, const gs_com2* lin_pi, const gs_com1* lin_theta, uint8_t* out_ok) {
  const bool set = a_consts && b_consts && gamma && tp && tq && xcoms && ycoms && pi && theta && lin_pi && lin_theta && out_ok;
  if (int rc = zk_args(ctx, "zk_ppe_verify", count, m, n, K, set)) return rc;
  if (count == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const zk_host h{m, n, K, a_consts, xcoms, ycoms, pi, theta, lin_pi, lin_theta};
  gs_com2 w2;
  if (int rc = crs_w2(ctx, &w2)) return rc;
  const size_t mk = m + K, chunk = zk_chunk(ctx, K);
  for (size_t off = 0; off < count; off += chunk) {
    const size_t cn = std::min(chunk, count - off), nl = cn * K;
    const zk_layout L(cn, m, n, K, b_consts + off * m, gamma + off * m * n, tp + off * K, tq + off * K);
    Scratch sc(ctx);
    zk_dev d;
    if (int rc = zk_upload(ctx, sc, h, L, w2, off, cn, &d)) return rc;
    gs_gt* dT;
    uint8_t *ok_ppe, *ok_lin, *dok;
    CUDA_TRY(upload(ctx, sc, &dT, L.ones.data(), cn));
    CUDA_TRY(sc.alloc(&ok_ppe, cn));
    CUDA_TRY(sc.alloc(&ok_lin, nl));
    CUDA_TRY(sc.alloc(&dok, cn));
    int rc = verify_dev(ctx, GS_PPE, cn, mk, n, d.A, d.B, (const gs_fr*)d.G, dT, d.c, d.d, d.pi, d.th, false, ok_ppe);
    if (rc) return rc;
    // every L_k has the y-commitment W2: its lines are walked once per pass
    rc = verify_dev(ctx, GS_MSMEG1, nl, 1, 1, d.La, d.Lb, (const gs_fr*)d.Lg, d.Lt, d.Lc, (const gs_com2*)d.Ld, d.Lpi, d.Lth, true,
                    ok_lin);
    if (rc) return rc;
    LAUNCH(k_zk_and, cn, ok_ppe, ok_lin, cn, (int)K, dok);
    CUDA_TRY(cudaMemcpyAsync(out_ok + off, dok, cn, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

int gs_zk_ppe_verify_each_rand(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                               const gs_g2* b_consts, const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq, const gs_com1* xcoms,
                               const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const gs_com2* lin_pi,
                               const gs_com1* lin_theta, const uint64_t* rho, uint8_t* out_ok) {
  const bool set =
      a_consts && b_consts && gamma && tp && tq && xcoms && ycoms && pi && theta && lin_pi && lin_theta && rho && out_ok;
  if (int rc = zk_args(ctx, "zk_ppe_verify_each_rand", count, m, n, K, set)) return rc;
  if (count == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  const zk_host h{m, n, K, a_consts, xcoms, ycoms, pi, theta, lin_pi, lin_theta};
  gs_com2 w2;
  if (int rc = crs_w2(ctx, &w2)) return rc;
  const size_t mk = m + K, chunk = zk_chunk(ctx, K);
  // rho: PPE' of statement i at 2i, L_k at 2 count + 2(iK + k), beta last
  const uint64_t *rho_lin = rho + 2 * count, *rho_beta = rho + 2 * count * (1 + K);
  for (size_t off = 0; off < count; off += chunk) {
    const size_t cn = std::min(chunk, count - off);
    const zk_layout L(cn, m, n, K, b_consts + off * m, gamma + off * m * n, tp + off * K, tq + off * K);
    Scratch sc(ctx);
    zk_dev d;
    uint8_t* dok;
    if (int rc = zk_upload(ctx, sc, h, L, w2, off, cn, &d)) return rc;
    CUDA_TRY(sc.alloc(&dok, cn));
    int rc = zk_each_rand_dev(ctx, cn, mk, n, K, (const gs_g1*)d.A, (const gs_g2*)d.B, (const gs_fr*)d.G, d.c, d.d, d.pi, d.th,
                              (const gs_g1*)d.La, (const gs_fr*)d.Lb, (const gs_fr*)d.Lg, (const gs_g1*)d.Lt, d.Lc,
                              (const gs_com2*)d.Ld, d.Lpi, d.Lth, rho + 2 * off, rho_lin + 2 * off * K, rho_beta, dok);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_ok + off, dok, cn, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

}  // extern "C"
