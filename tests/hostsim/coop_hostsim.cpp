// Host instantiation of the cooperative Fp12 ops (coop12.cuh) for tests/test_coop_reduce_hostsim.py.  Built twice: with
// the default dot-product forms and with -DGS_LINE_KARATSUBA=1 -DGS_MUL_KARATSUBA=1 (three reduced sums), so that the
// test can compare the two byte for byte.  Fp12 values cross the C ABI in tower order, Montgomery limbs.
#include <cstring>
#include <vector>
#include "../../groth-sahai-rs_b200/csrc/pairing.cuh"
#include "../../groth-sahai-rs_b200/csrc/coop12.cuh"
using namespace gs;

static void from_tower(uint32_t* acc, int lane, const fp12& x) {
  for (int k = 0; k < 6; k++) cq_st_coef(acc, k, lane, ((const fp2*)&x)[cq_tower_pos(k)]);
}
static void to_tower(fp12& x, const uint32_t* acc, int lane) {
  for (int k = 0; k < 6; k++) {
    fp2 c;
    cq_ld_coef(c.c0, c.c1, acc, k, lane, false, false);
    ((fp2*)&x)[cq_tower_pos(k)] = c;
  }
}

extern "C" {
// which forms this build runs (10 * GS_LINE_KARATSUBA + GS_MUL_KARATSUBA)
int hs_forms() { return 10 * GS_LINE_KARATSUBA + GS_MUL_KARATSUBA; }

// r = sum_{t<nt} Y_t X_t through cq_fp2_dot_w: y = nt Fp2 (c0, c1), x = nt Fp2, each operand in lane `lane` of the Q layout
void hs_dot_w(void* r, int nt, const void* y, const void* x, int lane) {
  const fp2* Y = (const fp2*)y;
  const fp2* X = (const fp2*)x;
  std::vector<uint32_t> q(8 * CQ_FP, 0xdeadbeefu);
  fp yr[8];
  const uint32_t *x0[4], *x1[4];
  for (int t = 0; t < nt; t++) {
    yr[2 * t] = Y[t].c0;
    yr[2 * t + 1] = Y[t].c1;
    cq_st(cq_ptr(q.data(), 2 * t, lane), X[t].c0);
    cq_st(cq_ptr(q.data(), 2 * t + 1, lane), X[t].c1);
    x0[t] = cq_ptr(q.data(), 2 * t, lane);
    x1[t] = cq_ptr(q.data(), 2 * t + 1, lane);
  }
  fp2 o;
  o.c0.set_zero();
  o.c1.set_zero();
#define DOT(NT)                                                         \
  case NT: {                                                            \
    fp yy[2 * NT];                                                      \
    const uint32_t *a0[NT], *a1[NT];                                    \
    for (int t = 0; t < NT; t++) {                                      \
      yy[2 * t] = yr[2 * t];                                            \
      yy[2 * t + 1] = yr[2 * t + 1];                                    \
      a0[t] = x0[t];                                                    \
      a1[t] = x1[t];                                                    \
    }                                                                   \
    cq_fp2_dot_w<NT>(o, cq_yreg<NT>{yy}, a0, a1);                       \
  } break;
  switch (nt) { DOT(1) DOT(2) DOT(3) DOT(4) default: break; }
#undef DOT
  memcpy(r, &o, sizeof(o));
}

// f * (alpha + beta w^2 + w^3) through cq_line_mul_u; tile = alpha.c0, alpha.c1, beta.c0, beta.c1
void hs_line_mul_u(void* r, const void* a, const void* tile4, int lane) {
  fp12 x;
  memcpy(&x, a, sizeof(x));
  const fp* T = (const fp*)tile4;
  std::vector<uint32_t> f(CQ_ACC, 0xdeadbeefu), o(CQ_ACC, 0xdeadbeefu), tile(4 * CQ_FP, 0xdeadbeefu);
  from_tower(f.data(), lane, x);
  for (int i = 0; i < 4; i++) cq_st(cq_ptr(tile.data(), i, lane), T[i]);
  for (int k = 0; k < 6; k++) cq_line_mul_u(k, lane, f.data(), o.data(), tile.data(), true);
  fp12 z;
  to_tower(z, o.data(), lane);
  memcpy(r, &z, sizeof(z));
}
void hs_sqr(void* r, const void* a, int lane) {
  fp12 x;
  memcpy(&x, a, sizeof(x));
  std::vector<uint32_t> f(CQ_ACC, 0xdeadbeefu), o(CQ_ACC, 0xdeadbeefu);
  from_tower(f.data(), lane, x);
  for (int k = 0; k < 6; k++) cq_sqr(k, lane, f.data(), o.data());
  fp12 z;
  to_tower(z, o.data(), lane);
  memcpy(r, &z, sizeof(z));
}
void hs_mul(void* r, const void* a, const void* b, int lane) {
  fp12 x, y;
  memcpy(&x, a, sizeof(x));
  memcpy(&y, b, sizeof(y));
  std::vector<uint32_t> f(CQ_ACC, 0xdeadbeefu), g(CQ_ACC, 0xdeadbeefu), o(CQ_ACC, 0xdeadbeefu);
  from_tower(f.data(), lane, x);
  from_tower(g.data(), lane, y);
  for (int k = 0; k < 6; k++) cq_mul(k, lane, f.data(), g.data(), o.data());
  fp12 z;
  to_tower(z, o.data(), lane);
  memcpy(r, &z, sizeof(z));
}

// the final-exponentiation op program (finalexp.cu)
void hs_final_exp(void* r, const void* a, int lane) {
  fp12 x;
  memcpy(&x, a, sizeof(x));
  std::vector<uint32_t> bufs(CQ_FE_NBUF * CQ_ACC, 0xdeadbeefu);
  from_tower(bufs.data(), lane, x);
  static uint32_t prog[CQ_FE_MAXOPS];
  const int n = cq_build_final_exp(prog);
  for (int i = 0; i < n; i++)
    for (int k = 0; k < 6; k++) cq_exec(prog[i], k, lane, bufs.data());
  fp12 z;
  to_tower(z, bufs.data() + CQ_FE_OUT * CQ_ACC, lane);
  memcpy(r, &z, sizeof(z));
}

// Miller loop of k_miller4 for one accumulator (lane) and n <= 4 pairs: the affine line walk (pairing.cuh) with
// unit-gamma line tiles, cq_sqr and cq_line_mul_u; conjugated at the end (x < 0).  Equals the projective Miller value
// up to subfield factors, i.e. after the final exponentiation.
void hs_miller(void* r, int n, const void* g1s, const void* g2s, int lane) {
  const g1_aff* P = (const g1_aff*)g1s;
  const g2_aff* Q = (const g2_aff*)g2s;
  fp2 Tx[4], Ty[4], Qx[4], Qy[4], lam[4], mu[4];
  bool act[4] = {false, false, false, false};
  fp s[4], w[4];
  for (int i = 0; i < n && i < 4; i++) {
    if (P[i].is_inf() || Q[i].is_inf()) continue;
    act[i] = true;
    Tx[i] = Q[i].x;
    Ty[i] = Q[i].y;
    Qx[i] = Q[i].x;
    Qy[i] = Q[i].y;
    fp_inv(w[i], P[i].y);
    fp::mul(s[i], P[i].x, w[i]);
    fp::neg(s[i], s[i]);
  }
  std::vector<uint32_t> acc(2 * CQ_ACC, 0xdeadbeefu), tile(4 * CQ_FP, 0xdeadbeefu);
  int cur = 0;
  for (int k = 0; k < 6; k++) cq_set_one(k, lane, acc.data());
  for (int bit = 62; bit >= 0; bit--) {
    if (bit != 62) {
      for (int k = 0; k < 6; k++) cq_sqr(k, lane, acc.data() + cur * CQ_ACC, acc.data() + (cur ^ 1) * CQ_ACC);
      cur ^= 1;
    }
    const int nl = ((GS_X_ABS >> bit) & 1) ? 2 : 1;
    for (int t = 0; t < nl; t++) {
      g2_pts_arr TT{Tx, Ty}, QQ{Qx, Qy};
      g2_affine_step<4>(TT, QQ, act, t == 1, [&](int i, const fp2& l, const fp2& m) { lam[i] = l; mu[i] = m; }, [] {});
      for (int i = 3; i >= 0; i--) {
        if (!act[i]) continue;
        fp v;
        fp::mul(v, mu[i].c0, w[i]);
        cq_st(cq_ptr(tile.data(), 0, lane), v);
        fp::mul(v, mu[i].c1, w[i]);
        cq_st(cq_ptr(tile.data(), 1, lane), v);
        fp::mul(v, lam[i].c0, s[i]);
        cq_st(cq_ptr(tile.data(), 2, lane), v);
        fp::mul(v, lam[i].c1, s[i]);
        cq_st(cq_ptr(tile.data(), 3, lane), v);
        for (int k = 0; k < 6; k++)
          cq_line_mul_u(k, lane, acc.data() + cur * CQ_ACC, acc.data() + (cur ^ 1) * CQ_ACC, tile.data(), true);
        cur ^= 1;
      }
    }
  }
  fp12 out;
  for (int k = 0; k < 6; k++) {
    fp2 c;
    cq_ld_coef(c.c0, c.c1, acc.data() + cur * CQ_ACC, k, lane, false, false);
    if (k & 1) fp2::neg(c, c);
    ((fp2*)&out)[cq_tower_pos(k)] = c;
  }
  memcpy(r, &out, sizeof(out));
}
}
