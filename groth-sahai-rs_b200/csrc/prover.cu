// Prover side of the C ABI: CRS generation, the four batch_commit_* variants, Provable::prove for the
// four equation types, Mat products.  The group-templated kernels live in prover_g1.cu / prover_g2.cu.
// Reference: src/generator.rs:81-118, src/prover/commit.rs:78-256, src/prover/prove.rs:92-488,
// src/data_structures.rs:645-742 / 768-913.
#include "ctx.h"
#include "endo.cuh"

using namespace gs;

namespace gs {

// ------------------------------------------------------------------ CRS
struct crs_gen_in {
  g1_aff p1;
  g2_aff p2;
  fr a1, a2, t1, t2;
};
struct crs_gen_out {
  g1_aff p1, q1, u1, v1;
  g2_aff p2, q2, u2, v2;
};
// generator.rs:96-109: q1 = a1 p1, u1 = t1 p1, v1 = t1 q1 = (t1 a1) p1 ; same on G2.
// Six scalar multiplications, each split along the group's endomorphism (endo.cuh: 2 x 128-bit parts on G1, 4 x 64-bit on
// G2) so that the serial chain is 32 / 16 windows instead of 64: thread t < 6 -> G1 product t / 2, part t % 2;
// thread 6 + t (t < 12) -> G2 product t / 4, part t % 4.  The parts are summed and normalised by thread 0 of each product.
__global__ void __launch_bounds__(32) k_crs_generate(const crs_gen_in* in, crs_gen_out* out) {
  __shared__ g1_jac p1s[6];
  __shared__ g2_jac p2s[12];
  const int t = threadIdx.x;
  if (blockIdx.x != 0) return;
  if (t < 18) {
    const bool g1side = t < 6;
    const int prod = g1side ? t / 2 : (t - 6) / 4, part = g1side ? t % 2 : (t - 6) % 4;
    fr s;
    if (prod == 0) s = g1side ? in->a1 : in->a2;
    if (prod == 1) s = g1side ? in->t1 : in->t2;
    if (prod == 2) {
      if (g1side)
        fr::mul(s, in->a1, in->t1);
      else
        fr::mul(s, in->a2, in->t2);
    }
    uint32_t k[8];
    fr_from_mont(k, s);
    if (g1side)
      EndoSplit<FpOps>::part(p1s[t], in->p1, k, part);
    else
      EndoSplit<Fp2Ops>::part(p2s[t - 6], in->p2, k, part);
  }
  __syncthreads();
  if (t < 3) {
    g1_jac j = p1s[2 * t];
    g1_jac::add(j, j, p1s[2 * t + 1]);
    g1_aff a;
    g1_jac::to_affine(a, j);
    if (t == 0) out->q1 = a;
    if (t == 1) out->u1 = a;
    if (t == 2) out->v1 = a;
    if (t == 0) out->p1 = in->p1;
  } else if (t >= 6 && t < 9) {
    const int q = t - 6;
    g2_jac j = p2s[4 * q];
    for (int i = 1; i < 4; i++) g2_jac::add(j, j, p2s[4 * q + i]);
    g2_aff a;
    g2_jac::to_affine(a, j);
    if (q == 0) out->q2 = a;
    if (q == 1) out->u2 = a;
    if (q == 2) out->v2 = a;
    if (q == 0) out->p2 = in->p2;
  }
}

// W1 = u2 + (O, g1), W2 = v2 + (O, g2), and the negations used by verify
__global__ void k_crs_derive(crs_dev* c) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  c->w1[0] = c->u[1][0];
  {
    g1_jac j;
    j.from_affine(c->u[1][1]);
    g1_jac::add_mixed(j, j, c->g1);
    g1_jac::to_affine(c->w1[1], j);
  }
  c->w2[0] = c->v[1][0];
  {
    g2_jac j;
    j.from_affine(c->v[1][1]);
    g2_jac::add_mixed(j, j, c->g2);
    g2_jac::to_affine(c->w2[1], j);
  }
  for (int k = 0; k < 2; k++)
    for (int a = 0; a < 2; a++) {
      c->neg_u[k][a] = c->u[k][a];
      fp::neg(c->neg_u[k][a].y, c->neg_u[k][a].y);
    }
  for (int a = 0; a < 2; a++) {
    c->neg_w1[a] = c->w1[a];
    fp::neg(c->neg_w1[a].y, c->neg_w1[a].y);
  }
}

// ------------------------------------------------------------------ Fr matrix algebra
// The three dot-product kernels below run with `lanes` = 1 (one thread per output: small statements, big batches) or
// `lanes` = 32 (one warp per output, strided partial sums + a shuffle tree: ONE big statement, where an output is a
// dot product over 1,024 .. 65,536 terms and there are only a handful of outputs).
__device__ GS_INL void fr_warp_sum(fr& acc) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    fr o;
#pragma unroll
    for (int i = 0; i < 8; i++) o.l[i] = __shfl_down_sync(0xffffffffu, acc.l[i], off);
    fr::add(acc, acc, o);
  }
}

// out (r x c) = A (r x k) * B (k x c), row-major; optional transposes via strides.
// Every prover kernel is batched over blockIdx.y = proof instance; `*_bs` = elements between instances (0: shared).
__global__ void k_fr_matmul(fr* __restrict__ out, const fr* __restrict__ A, size_t a_rs, size_t a_cs, const fr* __restrict__ B,
                            size_t b_rs, size_t b_cs, size_t r, size_t k, size_t c, size_t a_bs, size_t b_bs, int lanes) {
  size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t id = gid / lanes;
  const int lane = (int)(gid % lanes);
  if (id >= r * c) return;
  out += (size_t)blockIdx.y * r * c;
  A += (size_t)blockIdx.y * a_bs;
  B += (size_t)blockIdx.y * b_bs;
  size_t i = id / c, j = id % c;
  fr acc;
  acc.set_zero();
  for (size_t t = lane; t < k; t += lanes) {
    fr p;
    fr::mul(p, A[i * a_rs + t * a_cs], B[t * b_rs + j * b_cs]);
    fr::add(acc, acc, p);
  }
  if (lanes == 32) fr_warp_sum(acc);
  if (lane == 0) out[id] = acc;
}

// coef_pi[i][l] = (RG * S)[i][l] - T[l][i]            (prove.rs:139-142)   cx x cy
__global__ void k_coef_pi(fr* __restrict__ out, const fr* __restrict__ RG, const fr* __restrict__ S, const fr* __restrict__ T, int cx,
                          int cy, size_t n, size_t s_bs, int lanes) {
  int gid = blockIdx.x * blockDim.x + threadIdx.x;
  int id = gid / lanes;
  const int lane = gid % lanes;
  if (id >= cx * cy) return;
  out += (size_t)blockIdx.y * cx * cy;
  RG += (size_t)blockIdx.y * cx * n;
  S += (size_t)blockIdx.y * s_bs;
  T += (size_t)blockIdx.y * cx * cy;
  int i = id / cy, l = id % cy;
  fr acc;
  acc.set_zero();
  for (size_t j = lane; j < n; j += lanes) {
    fr p;
    fr::mul(p, RG[i * n + j], S[j * cy + l]);
    fr::add(acc, acc, p);
  }
  if (lanes == 32) fr_warp_sum(acc);
  if (lane != 0) return;
  fr::sub(acc, acc, T[l * cx + i]);
  out[id] = acc;
}

// scalar vectors of the variable-base part of a proof element:
//   sv[i][t] = R[t][i] (t < m) ; RG[i][t-m] (t >= m)          i < cx
__global__ void k_concat_scalars(fr* __restrict__ sv, const fr* __restrict__ R, const fr* __restrict__ RG, int cx, size_t m, size_t n,
                                 size_t r_bs) {
  size_t id = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= (size_t)cx * (m + n)) return;
  sv += (size_t)blockIdx.y * cx * (m + n);
  R += (size_t)blockIdx.y * r_bs;
  RG += (size_t)blockIdx.y * cx * n;
  size_t i = id / (m + n), t = id % (m + n);
  sv[id] = t < m ? R[t * cx + i] : RG[i * n + (t - m)];
}

// dot[i] = sum_t sv[i][t] * w[t]    (scalar-typed constants/variables: everything collapses onto W)
__global__ void k_fr_dot(fr* __restrict__ out, const fr* __restrict__ sv, const fr* __restrict__ w0, size_t m, const fr* __restrict__ w1,
                         size_t n, int rows, size_t w1_bs, int lanes) {
  int gid = blockIdx.x * blockDim.x + threadIdx.x;
  int i = gid / lanes;
  const int lane = gid % lanes;
  if (i >= rows) return;
  out += (size_t)blockIdx.y * rows;
  sv += (size_t)blockIdx.y * rows * (m + n);
  w0 += (size_t)blockIdx.y * m;
  w1 += (size_t)blockIdx.y * w1_bs;
  fr acc;
  acc.set_zero();
  for (size_t t = lane; t < m + n; t += lanes) {
    fr p;
    fr::mul(p, sv[(size_t)i * (m + n) + t], t < m ? w0[t] : w1[t - m]);
    fr::add(acc, acc, p);
  }
  if (lanes == 32) fr_warp_sum(acc);
  if (lane == 0) out[i] = acc;
}

}  // namespace gs

namespace gsi {
extern template int batch_commit_impl<FpOps>(gs_ctx*, size_t, int, int, const gs_fr*, size_t, const gs_fr*, size_t, size_t, const void*, void*);
extern template int batch_commit_impl<Fp2Ops>(gs_ctx*, size_t, int, int, const gs_fr*, size_t, const gs_fr*, size_t, size_t, const void*, void*);
extern template int com_matmul_impl<FpOps>(gs_ctx*, size_t, size_t, size_t, const gs_fr*, const void*, void*);
extern template int com_matmul_impl<Fp2Ops>(gs_ctx*, size_t, size_t, size_t, const gs_fr*, const void*, void*);

// generator.rs:96-109 on the device (6 scalar multiplications)
int crs_generate_points(gs_ctx* ctx, const gs_g1* p1, const gs_g2* p2, const gs_fr* a1, const gs_fr* a2, const gs_fr* t1,
                        const gs_fr* t2, gs_crs* out) {
  Scratch sc(ctx);
  crs_gen_in hin;
  memcpy(&hin.p1, p1, sizeof(g1_aff));
  memcpy(&hin.p2, p2, sizeof(g2_aff));
  memcpy(&hin.a1, a1, sizeof(fr));
  memcpy(&hin.a2, a2, sizeof(fr));
  memcpy(&hin.t1, t1, sizeof(fr));
  memcpy(&hin.t2, t2, sizeof(fr));
  crs_gen_in* din;
  crs_gen_out* dout;
  CUDA_TRY(upload(ctx, sc, &din, &hin, 1));
  CUDA_TRY(sc.alloc(&dout, 1));
  LAUNCH_CFG(k_crs_generate, 32, 32, 0, din, dout);
  crs_gen_out hout;
  CUDA_TRY(cudaMemcpyAsync(&hout, dout, sizeof(hout), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  memset(out, 0, sizeof(*out));
  memcpy(&out->u[0].p[0], &hout.p1, sizeof(g1_aff));
  memcpy(&out->u[0].p[1], &hout.q1, sizeof(g1_aff));
  memcpy(&out->u[1].p[0], &hout.u1, sizeof(g1_aff));
  memcpy(&out->u[1].p[1], &hout.v1, sizeof(g1_aff));
  memcpy(&out->v[0].p[0], &hout.p2, sizeof(g2_aff));
  memcpy(&out->v[0].p[1], &hout.q2, sizeof(g2_aff));
  memcpy(&out->v[1].p[0], &hout.u2, sizeof(g2_aff));
  memcpy(&out->v[1].p[1], &hout.v2, sizeof(g2_aff));
  out->g1_gen = *p1;
  out->g2_gen = *p2;
  return GS_OK;
}

int crs_derive(gs_ctx* ctx) {
  LAUNCH(k_crs_derive, 1, ctx->crs);
  return GS_OK;
}
}  // namespace gsi

using namespace gsi;

extern "C" {

int gs_batch_commit_g1(gs_ctx* ctx, size_t n, const gs_g1* xvars, const gs_fr* rand, gs_com1* out) {
  if (!xvars || !rand) return GS_EARG;
  return batch_commit_impl<FpOps>(ctx, n, /*u1*/ 0, /*u2*/ 1, rand, 2, rand + 1, 2, 2 * n, xvars, out);
}
int gs_batch_commit_g2(gs_ctx* ctx, size_t n, const gs_g2* yvars, const gs_fr* rand, gs_com2* out) {
  if (!yvars || !rand) return GS_EARG;
  return batch_commit_impl<Fp2Ops>(ctx, n, 0, 1, rand, 2, rand + 1, 2, 2 * n, yvars, out);
}
int gs_batch_commit_scalar_b1(gs_ctx* ctx, size_t n, const gs_fr* xs, const gs_fr* rand, gs_com1* out) {
  if (!xs || !rand || !ctx) return GS_EARG;
  // c_i = x_i W1 + r_i u1: pack [xs | rand] so that one upload serves both scalar streams
  std::vector<gs_fr> buf(2 * n);
  if (n) {
    memcpy(buf.data(), xs, n * sizeof(gs_fr));
    memcpy(buf.data() + n, rand, n * sizeof(gs_fr));
  }
  return batch_commit_impl<FpOps>(ctx, n, /*W1*/ 2, /*u1*/ 0, buf.data(), 1, buf.data() + n, 1, 2 * n, nullptr, out);
}
int gs_batch_commit_scalar_b2(gs_ctx* ctx, size_t n, const gs_fr* ys, const gs_fr* rand, gs_com2* out) {
  if (!ys || !rand || !ctx) return GS_EARG;
  std::vector<gs_fr> buf(2 * n);
  if (n) {
    memcpy(buf.data(), ys, n * sizeof(gs_fr));
    memcpy(buf.data() + n, rand, n * sizeof(gs_fr));
  }
  return batch_commit_impl<Fp2Ops>(ctx, n, 2, 0, buf.data(), 1, buf.data() + n, 1, 2 * n, nullptr, out);
}

}  // extern "C"

// `count` independent Provable::prove calls of one type and shape, every kernel batched over blockIdx.y.
// Per-proof arrays are contiguous ([count][...]); with shared_vars the witnesses and their commitment randomness
// are one set.  gs_prove is the batch of one.
int gsi::prove_impl(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                    const gs_fr* gamma, const void* xvars, const void* yvars, const gs_fr* x_rand, const gs_fr* y_rand,
                    const gs_fr* pf_rand, bool shared_vars, gs_com2* out_pi, gs_com1* out_theta) {
  if (!ctx) return GS_EARG;
  if (type < 0 || type > 3) FAIL(GS_EARG, "prove: bad equation type");
  if (!ctx->crs_loaded) FAIL(GS_EARG, "prove: no CRS loaded");
  if (count == 0) return GS_OK;
  if (m == 0 || n == 0) FAIL(GS_EDIM, "prove: empty variable list");  // reference panics (SURVEY.md §3.7)
  if (m > 1 << 22 || n > 1 << 22) FAIL(GS_EDIM, "prove: too many variables");
  if (!a_consts || !b_consts || !gamma || !xvars || !yvars || !x_rand || !y_rand || !pf_rand || !out_pi || !out_theta)
    return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  const int cx = s.cx, cy = s.cy;
  const size_t szA = elem_size_A(type), szB = elem_size_B(type);
  const size_t MAXB = 32768;  // gridDim.y limit is 65,535
  for (size_t off = 0; off < count; off += MAXB) {
    const size_t nb = count - off < MAXB ? count - off : MAXB;
    const size_t voff = shared_vars ? 0 : off, nv = shared_vars ? 1 : nb;
    Scratch sc(ctx);
    uint8_t *dA, *dB, *dX, *dY;
    fr *dG, *dR, *dS, *dT;
    CUDA_TRY(upload(ctx, sc, &dA, (const char*)a_consts + off * n * szA, nb * n * szA));
    CUDA_TRY(upload(ctx, sc, &dB, (const char*)b_consts + off * m * szB, nb * m * szB));
    CUDA_TRY(upload(ctx, sc, &dX, (const char*)xvars + voff * m * szA, nv * m * szA));
    CUDA_TRY(upload(ctx, sc, &dY, (const char*)yvars + voff * n * szB, nv * n * szB));
    CUDA_TRY(upload(ctx, sc, &dG, gamma + off * m * n, nb * m * n));
    CUDA_TRY(upload(ctx, sc, &dR, x_rand + voff * m * cx, nv * m * cx));
    CUDA_TRY(upload(ctx, sc, &dS, y_rand + voff * n * cy, nv * n * cy));
    CUDA_TRY(upload(ctx, sc, &dT, pf_rand + off * cx * cy, nb * cx * cy));
    const size_t r_bs = shared_vars ? 0 : m * cx, s_bs = shared_vars ? 0 : n * cy;  // instance strides of R, S
    fr *RG, *SG, *coef_pi, *sv_pi, *sv_th;
    CUDA_TRY(sc.alloc(&RG, nb * cx * n));
    CUDA_TRY(sc.alloc(&SG, nb * cy * m));
    CUDA_TRY(sc.alloc(&coef_pi, nb * cx * cy));
    CUDA_TRY(sc.alloc(&sv_pi, nb * cx * (m + n)));
    CUDA_TRY(sc.alloc(&sv_th, nb * cy * (m + n)));
    // RG = R^T Gamma (cx x n)  prove.rs:133 ;  SG = S^T Gamma^T (cy x m)  prove.rs:154
    const int l_rg = fr_lanes(m, (size_t)cx * n * nb), l_sg = fr_lanes(n, (size_t)cy * m * nb), l_cp = fr_lanes(n, (size_t)cx * cy * nb);
    LAUNCH_B(k_fr_matmul, (size_t)cx * n * l_rg, nb, RG, dR, (size_t)1, (size_t)cx, dG, n, (size_t)1, (size_t)cx, m, n, r_bs, m * n, l_rg);
    LAUNCH_B(k_fr_matmul, (size_t)cy * m * l_sg, nb, SG, dS, (size_t)1, (size_t)cy, dG, (size_t)1, n, (size_t)cy, n, m, s_bs, m * n, l_sg);
    // (R^T Gamma S - T^T)  prove.rs:139-142
    LAUNCH_B(k_coef_pi, (size_t)cx * cy * l_cp, nb, coef_pi, RG, dS, dT, cx, cy, n, s_bs, l_cp);
    LAUNCH_B(k_concat_scalars, (size_t)cx * (m + n), nb, sv_pi, dR, RG, cx, m, n, r_bs);
    LAUNCH_B(k_concat_scalars, (size_t)cy * (m + n), nb, sv_th, dS, SG, cy, n, m, s_bs);
    g2_aff* dpi;
    g1_aff* dth;
    CUDA_TRY(sc.alloc(&dpi, nb * 2 * cx));
    CUDA_TRY(sc.alloc(&dth, nb * 2 * cy));
    // pi_i = sum_k R[k][i] iota(B_k) + sum_j RG[i][j] iota(Y_j) + sum_l coef_pi[i][l] v_l        (l < cy)
    fr *e_pi = nullptr, *e_th = nullptr;
    if (!s.groupB) {  // scalar-typed y side: every term collapses onto W2
      CUDA_TRY(sc.alloc(&e_pi, nb * cx));
      const int l_d = fr_lanes(m + n, (size_t)cx * nb);
      LAUNCH_B(k_fr_dot, (size_t)cx * l_d, nb, e_pi, sv_pi, (const fr*)dB, m, (const fr*)dY, n, cx, shared_vars ? (size_t)0 : n, l_d);
    }
    if (!s.groupA) {
      CUDA_TRY(sc.alloc(&e_th, nb * cy));
      const int l_d = fr_lanes(m + n, (size_t)cy * nb);
      LAUNCH_B(k_fr_dot, (size_t)cy * l_d, nb, e_th, sv_th, (const fr*)dA, n, (const fr*)dX, m, cy, shared_vars ? (size_t)0 : m, l_d);
    }
    // theta_i = sum_j S[j][i] iota(A_j) + sum_k SG[i][k] iota(X_k) + sum_l T[i][l] u_l          (l < cx)
    // theta on the second stream next to pi in the latency regime (few proofs)
    int rc = theta_pi_fork(
        ctx, nb * (m + n) * 2 < 32768,
        [&] { return proof_element<FpOps>(ctx, sc, nb, cy, s.groupA, sv_th, dA, n, dX, m, shared_vars, cx, dT, (size_t)cx, e_th, dth); },
        [&] {
          return proof_element<Fp2Ops>(ctx, sc, nb, cx, s.groupB, sv_pi, dB, m, dY, n, shared_vars, cy, coef_pi, (size_t)cy, e_pi, dpi);
        });
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_pi + off * cx, dpi, nb * 2 * cx * sizeof(g2_aff), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_theta + off * cy, dth, nb * 2 * cy * sizeof(g1_aff), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  return GS_OK;
}

extern "C" {

int gs_prove(gs_ctx* ctx, int type, size_t m, size_t n, const void* a_consts, const void* b_consts, const gs_fr* gamma,
             const void* xvars, const void* yvars, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand,
             gs_com2* out_pi, gs_com1* out_theta) {
  return prove_impl(ctx, type, 1, m, n, a_consts, b_consts, gamma, xvars, yvars, x_rand, y_rand, pf_rand, false, out_pi, out_theta);
}

int gs_prove_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                   const gs_fr* gamma, const void* xvars, const void* yvars, const gs_fr* x_rand, const gs_fr* y_rand,
                   const gs_fr* pf_rand, int shared_vars, gs_com2* out_pi, gs_com1* out_theta) {
  return prove_impl(ctx, type, count, m, n, a_consts, b_consts, gamma, xvars, yvars, x_rand, y_rand, pf_rand, shared_vars != 0,
                    out_pi, out_theta);
}

}  // extern "C"

// `count` rerandomisations of committed proofs, laid out as prove_impl's arrays (shared_coms: one set of commitments and
// of R', S' for every equation).  With fresh R', S', T':
//   c' = c + R' u_x                     d' = d + S' v_y
//   pi'    = pi    + R'^T iota_y(B) + (R'^T Gamma) d + (R'^T Gamma S' - T'^T) v_y
//   theta' = theta + S'^T iota_x(A) + (S'^T Gamma^T) c + T' u_x
// -- exactly commit_and_prove of the same witnesses under R + R', S + S', T + T' + S'^T Gamma^T R.  The Fr algebra is
// prove_impl's; the variable-base sums run over the commitments (both coordinates) instead of iota(variables).
int gsi::rerandomize_impl(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                          const gs_fr* gamma, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                          const gs_com1* theta, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, bool shared,
                          gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta) {
  if (!ctx) return GS_EARG;
  if (type < 0 || type > 3) FAIL(GS_EARG, "rerandomize: bad equation type");
  if (!ctx->crs_loaded) FAIL(GS_EARG, "rerandomize: no CRS loaded");
  if (count == 0) return GS_OK;
  if (m == 0 || n == 0) FAIL(GS_EDIM, "rerandomize: empty variable list");
  if (m > 1 << 22 || n > 1 << 22) FAIL(GS_EDIM, "rerandomize: too many variables");
  if (!a_consts || !b_consts || !gamma || !xcoms || !ycoms || !pi || !theta || !x_rand || !y_rand || !pf_rand || !out_xcoms ||
      !out_ycoms || !out_pi || !out_theta)
    return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  verify_shape s = make_verify_shape(type, (int)m, (int)n);
  const int cx = s.cx, cy = s.cy;
  const size_t szA = elem_size_A(type), szB = elem_size_B(type);
  const size_t MAXB = 32768;  // gridDim.y limit is 65,535
  for (size_t off = 0; off < count; off += MAXB) {
    const size_t nb = count - off < MAXB ? count - off : MAXB;
    const size_t voff = shared ? 0 : off, nv = shared ? 1 : nb;
    Scratch sc(ctx);
    uint8_t *dA, *dB;
    fr *dG, *dR, *dS, *dT;
    g1_aff *dXc, *dTh;
    g2_aff *dYc, *dPi;
    CUDA_TRY(upload(ctx, sc, &dA, (const char*)a_consts + off * n * szA, nb * n * szA));
    CUDA_TRY(upload(ctx, sc, &dB, (const char*)b_consts + off * m * szB, nb * m * szB));
    CUDA_TRY(upload(ctx, sc, &dG, gamma + off * m * n, nb * m * n));
    CUDA_TRY(upload(ctx, sc, &dXc, xcoms + voff * m, nv * m * 2));
    CUDA_TRY(upload(ctx, sc, &dYc, ycoms + voff * n, nv * n * 2));
    CUDA_TRY(upload(ctx, sc, &dPi, pi + off * cx, nb * cx * 2));
    CUDA_TRY(upload(ctx, sc, &dTh, theta + off * cy, nb * cy * 2));
    CUDA_TRY(upload(ctx, sc, &dR, x_rand + voff * m * cx, nv * m * cx));
    CUDA_TRY(upload(ctx, sc, &dS, y_rand + voff * n * cy, nv * n * cy));
    CUDA_TRY(upload(ctx, sc, &dT, pf_rand + off * cx * cy, nb * cx * cy));
    // the new commitments (once for a shared set), on the main stream before the proof elements fork: a first call under
    // a key may (re)build the fixed-base tables that the elements read
    const bool do_coms = !shared || off == 0;
    g1_aff* dXo = nullptr;
    g2_aff* dYo = nullptr;
    if (do_coms) {
      CUDA_TRY(sc.alloc(&dXo, nv * m * 2));
      CUDA_TRY(sc.alloc(&dYo, nv * n * 2));
      int rc = rerand_commit<FpOps>(ctx, nv * m, cx, dR, dXc, dXo);
      if (rc) return rc;
      rc = rerand_commit<Fp2Ops>(ctx, nv * n, cy, dS, dYc, dYo);
      if (rc) return rc;
    }
    const size_t r_bs = shared ? 0 : m * cx, s_bs = shared ? 0 : n * cy;  // instance strides of R', S'
    fr *RG, *SG, *coef_pi, *sv_pi, *sv_th;
    CUDA_TRY(sc.alloc(&RG, nb * cx * n));
    CUDA_TRY(sc.alloc(&SG, nb * cy * m));
    CUDA_TRY(sc.alloc(&coef_pi, nb * cx * cy));
    CUDA_TRY(sc.alloc(&sv_pi, nb * cx * (m + n)));
    CUDA_TRY(sc.alloc(&sv_th, nb * cy * (m + n)));
    // RG = R'^T Gamma (cx x n), SG = S'^T Gamma^T (cy x m), coef_pi = R'^T Gamma S' - T'^T: as in prove_impl
    const int l_rg = fr_lanes(m, (size_t)cx * n * nb), l_sg = fr_lanes(n, (size_t)cy * m * nb), l_cp = fr_lanes(n, (size_t)cx * cy * nb);
    LAUNCH_B(k_fr_matmul, (size_t)cx * n * l_rg, nb, RG, dR, (size_t)1, (size_t)cx, dG, n, (size_t)1, (size_t)cx, m, n, r_bs, m * n, l_rg);
    LAUNCH_B(k_fr_matmul, (size_t)cy * m * l_sg, nb, SG, dS, (size_t)1, (size_t)cy, dG, (size_t)1, n, (size_t)cy, n, m, s_bs, m * n, l_sg);
    LAUNCH_B(k_coef_pi, (size_t)cx * cy * l_cp, nb, coef_pi, RG, dS, dT, cx, cy, n, s_bs, l_cp);
    LAUNCH_B(k_concat_scalars, (size_t)cx * (m + n), nb, sv_pi, dR, RG, cx, m, n, r_bs);
    LAUNCH_B(k_concat_scalars, (size_t)cy * (m + n), nb, sv_th, dS, SG, cy, n, m, s_bs);
    // scalar-typed constants collapse onto W: e_i = sum_k R'[k][i] b_k (pi'), sum_j S'[j][i] a_j (theta')
    fr *e_pi = nullptr, *e_th = nullptr;
    if (!s.groupB) {
      fr* rt;
      CUDA_TRY(sc.alloc(&rt, nb * cx * m));
      CUDA_TRY(sc.alloc(&e_pi, nb * cx));
      const int l_d = fr_lanes(m, (size_t)cx * nb);
      LAUNCH_B(k_concat_scalars, (size_t)cx * m, nb, rt, dR, RG, cx, m, (size_t)0, r_bs);
      LAUNCH_B(k_fr_dot, (size_t)cx * l_d, nb, e_pi, rt, (const fr*)dB, m, (const fr*)nullptr, (size_t)0, cx, (size_t)0, l_d);
    }
    if (!s.groupA) {
      fr* st;
      CUDA_TRY(sc.alloc(&st, nb * cy * n));
      CUDA_TRY(sc.alloc(&e_th, nb * cy));
      const int l_d = fr_lanes(n, (size_t)cy * nb);
      LAUNCH_B(k_concat_scalars, (size_t)cy * n, nb, st, dS, SG, cy, n, (size_t)0, s_bs);
      LAUNCH_B(k_fr_dot, (size_t)cy * l_d, nb, e_th, st, (const fr*)dA, n, (const fr*)nullptr, (size_t)0, cy, (size_t)0, l_d);
    }
    g2_aff* dpo;
    g1_aff* dto;
    CUDA_TRY(sc.alloc(&dpo, nb * 2 * cx));
    CUDA_TRY(sc.alloc(&dto, nb * 2 * cy));
    // theta' on the second stream next to pi' in the latency regime, as in prove_impl
    int rc = theta_pi_fork(
        ctx, nb * (m + n) * 2 < 32768,
        [&] { return rerand_element<FpOps>(ctx, sc, nb, cy, s.groupA, sv_th, SG, dA, n, dXc, m, shared, cx, dT, e_th, dTh, dto); },
        [&] { return rerand_element<Fp2Ops>(ctx, sc, nb, cx, s.groupB, sv_pi, RG, dB, m, dYc, n, shared, cy, coef_pi, e_pi, dPi, dpo); });
    if (rc) return rc;
    if (do_coms) {
      CUDA_TRY(cudaMemcpyAsync(out_xcoms + voff * m, dXo, nv * m * 2 * sizeof(g1_aff), cudaMemcpyDeviceToHost, ctx->stream));
      CUDA_TRY(cudaMemcpyAsync(out_ycoms + voff * n, dYo, nv * n * 2 * sizeof(g2_aff), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CUDA_TRY(cudaMemcpyAsync(out_pi + off * cx, dpo, nb * 2 * cx * sizeof(g2_aff), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(out_theta + off * cy, dto, nb * 2 * cy * sizeof(g1_aff), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  }
  return GS_OK;
}

extern "C" {

int gs_rerandomize(gs_ctx* ctx, int type, size_t m, size_t n, const void* a_consts, const void* b_consts, const gs_fr* gamma,
                   const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const gs_fr* x_rand,
                   const gs_fr* y_rand, const gs_fr* pf_rand, gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi,
                   gs_com1* out_theta) {
  return rerandomize_impl(ctx, type, 1, m, n, a_consts, b_consts, gamma, xcoms, ycoms, pi, theta, x_rand, y_rand, pf_rand, false,
                          out_xcoms, out_ycoms, out_pi, out_theta);
}

int gs_rerandomize_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                         const gs_fr* gamma, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta,
                         const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, int shared_coms, gs_com1* out_xcoms,
                         gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta) {
  return rerandomize_impl(ctx, type, count, m, n, a_consts, b_consts, gamma, xcoms, ycoms, pi, theta, x_rand, y_rand, pf_rand,
                          shared_coms != 0, out_xcoms, out_ycoms, out_pi, out_theta);
}

int gs_com1_matmul(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* lhs, const gs_com1* mat, gs_com1* out) {
  return com_matmul_impl<FpOps>(ctx, r, k, c, lhs, mat, out);
}
int gs_com2_matmul(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* lhs, const gs_com2* mat, gs_com2* out) {
  return com_matmul_impl<Fp2Ops>(ctx, r, k, c, lhs, mat, out);
}
int gs_fr_matmul(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* a, const gs_fr* b, gs_fr* out) {
  if (!ctx || !a || !b || !out) return GS_EARG;
  if (r == 0 || k == 0 || c == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  Scratch sc(ctx);
  fr *da, *db, *dout;
  CUDA_TRY(upload(ctx, sc, &da, a, r * k));
  CUDA_TRY(upload(ctx, sc, &db, b, k * c));
  CUDA_TRY(sc.alloc(&dout, r * c));
  const int l_mm = fr_lanes(k, r * c);
  LAUNCH(k_fr_matmul, r * c * l_mm, dout, da, k, (size_t)1, db, c, (size_t)1, r, k, c, (size_t)0, (size_t)0, l_mm);
  CUDA_TRY(cudaMemcpyAsync(out, dout, r * c * sizeof(fr), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return GS_OK;
}

}  // extern "C"
