// Zero-knowledge simulation with the hiding key's trapdoor (not in the reference): gs_simulate_batch makes accepting
// proofs without witnesses (Groth & Sahai, EUROCRYPT 2008, PAPERS.md).  Under the hiding key of gs_crs_generate's draws,
// W1 = u[1] + iota_1(g1) = t1 u[0] and W2 = t2 v[0], so the target of an equation can be absorbed into the proof through
// t1 / t2.  The simulator is the prover with every witness set to O / 0 (the SG and RG variable terms vanish):
//   c = R u_x                      d = S v_y
//   pi    = R^T iota_y(B) + (R^T Gamma S - T^T) v_y  (- t1 iota_2(T2)        MSMEG2)
//   theta = S^T iota_x(A) + T u_x                    (- t2 iota_1(T1)        MSMEG1;   - t t2 W1   Quad)
// PPE targets must be 1.  Each correction is one more constant column: a per-equation base (the target) with one
// scalar for the whole call (-t2 or -t1), or on a scalar-typed side one more term of the W coefficient.  This is the
// reference-order prove of an augmented equation with zero witnesses and one extra public variable whose commitment is
// W2 (W1): a commitment of 0 with randomness t2 (t1).  Every kernel is the prover's.
#include <cstddef>

#include "ctx.h"

using namespace gs;
using namespace gsi;

namespace {

// W = t key[0] for both coordinates: "extracting" the pairs (key[0].a, W.a) with t (k_extract, a = 0, 1) gives the identity
// twice.  `key0` = u[0] (v[0]) and `w` = W1 (W2), two device points each.
template <class F>
int trapdoor_matches(gs_ctx* ctx, const Aff<F>* key0, const Aff<F>* w, const gs_fr* t, bool* ok) {
  Scratch sc(ctx);
  Aff<F>* pairs;
  CUDA_TRY(sc.alloc(&pairs, 4));
  const size_t A = sizeof(Aff<F>);
  CUDA_TRY(cudaMemcpy2DAsync(pairs, 2 * A, key0, A, A, 2, cudaMemcpyDeviceToDevice, ctx->stream));
  CUDA_TRY(cudaMemcpy2DAsync(pairs + 1, 2 * A, w, A, A, 2, cudaMemcpyDeviceToDevice, ctx->stream));
  return extract_all_identity<F>(ctx, pairs, 2, t, ok);
}

}  // namespace

// tkey = (t1, t2) is the loaded CRS's simulation key iff W1 = t1 u[0] and W2 = t2 v[0].  Under a binding key
// W1 = t1 u[0] + iota_1(g1), so no key passes.  A validated key is cached until the next gs_crs_load / gs_crs_generate.
int gsi::sim_key_check(gs_ctx* ctx, const gs_fr* tkey) {
  if (ctx->tkey_valid && memcmp(ctx->tkey, tkey, sizeof(ctx->tkey)) == 0) return GS_OK;
  bool ok1, ok2;
  int rc = trapdoor_matches<FpOps>(ctx, &ctx->crs->u[0][0], &ctx->crs->w1[0], &tkey[0], &ok1);
  if (rc) return rc;
  rc = trapdoor_matches<Fp2Ops>(ctx, &ctx->crs->v[0][0], &ctx->crs->w2[0], &tkey[1], &ok2);
  if (rc) return rc;
  if (!ok1 || !ok2) FAIL(GS_EARG, "simulate: tkey is not the simulation key of the loaded CRS (t1, t2 of a hiding CRS)");
  memcpy(ctx->tkey, tkey, sizeof(ctx->tkey));
  ctx->tkey_valid = true;
  return GS_OK;
}

namespace {

// c_i = R[i] key for N commitments of O / 0 (host arrays): R[i][0] key_0 + R[i][1] key_1 (ns = 2) or r_i key_0 (ns = 1,
// the second scalar stream is a zero with stride 0 on W)
template <class F>
int commit_zero(gs_ctx* ctx, size_t N, int ns, const gs_fr* rand, void* out) {
  if (ns == 2) return batch_commit_impl<F>(ctx, N, 0, 1, rand, 2, rand + 1, 2, 2 * N, nullptr, out);
  std::vector<gs_fr> buf(N + 1);
  memcpy(buf.data(), rand, N * sizeof(gs_fr));
  return batch_commit_impl<F>(ctx, N, 0, 2, buf.data(), 1, buf.data() + N, 0, N + 1, nullptr, out);
}

// dst[i] = (src[i][0..n) | col[i]) for nb rows of elements of `sz` bytes (host -> device): the constants of an equation
// followed by its target
cudaError_t upload_with_column(gs_ctx* ctx, Scratch& sc, uint8_t** dst, const void* src, size_t n, const void* col, size_t nb,
                               size_t sz) {
  cudaError_t e = sc.alloc(dst, nb * (n + 1) * sz);
  if (e == cudaSuccess) e = cudaMemcpy2DAsync(*dst, (n + 1) * sz, src, n * sz, n * sz, nb, cudaMemcpyHostToDevice, ctx->stream);
  if (e == cudaSuccess)
    e = cudaMemcpy2DAsync(*dst + n * sz, (n + 1) * sz, col, sz, sz, nb, cudaMemcpyHostToDevice, ctx->stream);
  return e;
}

}  // namespace

int gsi::simulate_impl(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                       const gs_fr* gamma, const void* target, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, bool shared,
                       const gs_fr* tkey, gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta,
                       bool with_coms) {
  if (!ctx) return GS_EARG;
  if (type < 0 || type > 3) FAIL(GS_EARG, "simulate: bad equation type");
  if (!ctx->crs_loaded) FAIL(GS_EARG, "simulate: no CRS loaded");
  if (count == 0) return GS_OK;
  if (m == 0 || n == 0) FAIL(GS_EDIM, "simulate: empty variable list");
  if (m > 1 << 22 || n > 1 << 22) FAIL(GS_EDIM, "simulate: too many variables");
  if (!a_consts || !b_consts || !gamma || !target || !x_rand || !y_rand || !pf_rand || !tkey || (with_coms && (!out_xcoms || !out_ycoms)) ||
      !out_pi || !out_theta)
    return GS_EARG;
  if (type == GS_PPE) {
    fp12 one;
    one.set_one();
    for (size_t i = 0; i < count; i++)
      if (memcmp((const fp12*)target + i, &one, sizeof(fp12)) != 0)
        FAIL(GS_EARG, "simulate: a PPE target other than 1 has no simulated proof");
  }
  CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = sim_key_check(ctx, tkey);
  if (rc) return rc;
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  const int cx = s.cx, cy = s.cy;
  const size_t szA = elem_size_A(type), szB = elem_size_B(type), szT = elem_size_T(type);
  const size_t nv = shared ? 1 : count;
  // the commitments first: a big batch (re)builds the fixed-base tables that the proof elements read
  if (with_coms && (rc = commit_zero<FpOps>(ctx, nv * m, cx, x_rand, out_xcoms))) return rc;
  if (with_coms && (rc = commit_zero<Fp2Ops>(ctx, nv * n, cy, y_rand, out_ycoms))) return rc;
  // the extra constant column: theta's for MSMEG1 / Quad, pi's for MSMEG2, with the scalar -t2 / -t1 in every proof
  const size_t xa = (type == GS_MSMEG1 || type == GS_QUAD) ? 1 : 0, yb = type == GS_MSMEG2 ? 1 : 0;
  const size_t MAXB = 32768;  // gridDim.y limit is 65,535
  std::vector<gs_fr> negt;
  if (xa + yb) {
    fr t, nt;
    memcpy(&t, &tkey[yb ? 0 : 1], sizeof(fr));
    fr::neg(nt, t);
    negt.resize(count < MAXB ? count : MAXB);
    for (gs_fr& v : negt) memcpy(&v, &nt, sizeof(fr));
  }
  for (size_t off = 0; off < count; off += MAXB) {
    const size_t nb = count - off < MAXB ? count - off : MAXB;
    const size_t voff = shared ? 0 : off, nr = shared ? 1 : nb;
    Scratch sc(ctx);
    uint8_t *dA, *dB;
    fr *dG, *dR, *dS, *dT, *dneg = nullptr, *dtq = nullptr;
    const char* tgt = (const char*)target + off * szT;
    // a group-typed corrected side gets its target as constant n (m); Quad's target joins the W coefficient of theta
    if (s.groupA && xa)
      CUDA_TRY(upload_with_column(ctx, sc, &dA, (const char*)a_consts + off * n * szA, n, tgt, nb, szA));
    else
      CUDA_TRY(upload(ctx, sc, &dA, (const char*)a_consts + off * n * szA, nb * n * szA));
    if (yb)
      CUDA_TRY(upload_with_column(ctx, sc, &dB, (const char*)b_consts + off * m * szB, m, tgt, nb, szB));
    else
      CUDA_TRY(upload(ctx, sc, &dB, (const char*)b_consts + off * m * szB, nb * m * szB));
    if (type == GS_QUAD) CUDA_TRY(upload(ctx, sc, &dtq, tgt, nb));
    if (xa + yb) CUDA_TRY(upload(ctx, sc, &dneg, negt.data(), nb));
    CUDA_TRY(upload(ctx, sc, &dG, gamma + off * m * n, nb * m * n));
    CUDA_TRY(upload(ctx, sc, &dR, x_rand + voff * m * cx, nr * m * cx));
    CUDA_TRY(upload(ctx, sc, &dS, y_rand + voff * n * cy, nr * n * cy));
    CUDA_TRY(upload(ctx, sc, &dT, pf_rand + off * cx * cy, nb * cx * cy));
    const size_t r_bs = shared ? 0 : m * cx, s_bs = shared ? 0 : n * cy;  // instance strides of R, S
    // RG = R^T Gamma (cx x n) and coef_pi = R^T Gamma S - T^T, as in prove_impl
    fr *RG, *coef_pi, *sv_pi, *sv_th;
    CUDA_TRY(sc.alloc(&RG, nb * cx * n));
    CUDA_TRY(sc.alloc(&coef_pi, nb * cx * cy));
    CUDA_TRY(sc.alloc(&sv_pi, nb * cx * (m + yb)));
    CUDA_TRY(sc.alloc(&sv_th, nb * cy * (n + xa)));
    const int l_rg = fr_lanes(m, (size_t)cx * n * nb), l_cp = fr_lanes(n, (size_t)cx * cy * nb);
    LAUNCH_B(k_fr_matmul, (size_t)cx * n * l_rg, nb, RG, dR, (size_t)1, (size_t)cx, dG, n, (size_t)1, (size_t)cx, m, n, r_bs, m * n, l_rg);
    LAUNCH_B(k_coef_pi, (size_t)cx * cy * l_cp, nb, coef_pi, RG, dS, dT, cx, cy, n, s_bs, l_cp);
    // scalar rows: sv_pi[i] = (R[.][i] | -t1), sv_th[i] = (S[.][i] | -t2), the extra column only where a target is absorbed
    LAUNCH_B(k_concat_scalars, (size_t)cx * (m + yb), nb, sv_pi, dR, dneg, cx, m, yb, r_bs);
    LAUNCH_B(k_concat_scalars, (size_t)cy * (n + xa), nb, sv_th, dS, dneg, cy, n, xa, s_bs);
    // scalar-typed sides collapse onto W: e_i = sum_k R[k][i] b_k (pi), sum_j S[j][i] a_j (- t2 t on Quad) (theta)
    fr *e_pi = nullptr, *e_th = nullptr;
    if (!s.groupB) {
      CUDA_TRY(sc.alloc(&e_pi, nb * cx));
      const int l_d = fr_lanes(m, (size_t)cx * nb);
      LAUNCH_B(k_fr_dot, (size_t)cx * l_d, nb, e_pi, sv_pi, (const fr*)dB, m, (const fr*)nullptr, (size_t)0, cx, (size_t)0, l_d);
    }
    if (!s.groupA) {
      CUDA_TRY(sc.alloc(&e_th, nb * cy));
      const int l_d = fr_lanes(n + xa, (size_t)cy * nb);
      LAUNCH_B(k_fr_dot, (size_t)cy * l_d, nb, e_th, sv_th, (const fr*)dA, n, (const fr*)dtq, xa, cy, xa, l_d);
    }
    g2_aff* dpi;
    g1_aff* dth;
    CUDA_TRY(sc.alloc(&dpi, nb * 2 * cx));
    CUDA_TRY(sc.alloc(&dth, nb * 2 * cy));
    // proof_element without variable terms; theta on the second stream next to pi in the latency regime, as in prove_impl
    rc = theta_pi_fork(
        ctx, nb * (m + n) * 2 < 32768,
        [&] {
          return proof_element<FpOps>(ctx, sc, nb, cy, s.groupA, sv_th, dA, n + xa, nullptr, 0, shared, cx, dT, (size_t)cx, e_th, dth);
        },
        [&] {
          return proof_element<Fp2Ops>(ctx, sc, nb, cx, s.groupB, sv_pi, dB, m + yb, nullptr, 0, shared, cy, coef_pi, (size_t)cy, e_pi,
                                       dpi);
        });
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_pi + off * cx, dpi, nb * 2 * cx * sizeof(g2_aff), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_theta + off * cy, dth, nb * 2 * cy * sizeof(g1_aff), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  return GS_OK;
}

extern "C" {

int gs_simulate(gs_ctx* ctx, int type, size_t m, size_t n, const void* a_consts, const void* b_consts, const gs_fr* gamma,
                const void* target, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, const gs_fr* tkey,
                gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta) {
  return simulate_impl(ctx, type, 1, m, n, a_consts, b_consts, gamma, target, x_rand, y_rand, pf_rand, false, tkey, out_xcoms,
                       out_ycoms, out_pi, out_theta);
}

int gs_simulate_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                      const gs_fr* gamma, const void* target, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand,
                      int shared_coms, const gs_fr* tkey, gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi,
                      gs_com1* out_theta) {
  return simulate_impl(ctx, type, count, m, n, a_consts, b_consts, gamma, target, x_rand, y_rand, pf_rand, shared_coms != 0, tkey,
                       out_xcoms, out_ycoms, out_pi, out_theta);
}

}  // extern "C"
