// Extraction with the binding key (not in the reference): gs_extract opens commitments with the trapdoor a1 / a2 of
// gs_crs_generate.  Under the binding key u = [(p1, a1 p1), t1 (p1, a1 p1)] every commitment has c.1 = X + a1 c.0, so
// X = c.1 - a1 c.0 (ElGamal decryption); scalar commitments give x g1, the G2 side likewise with a2 (Groth & Sahai,
// EUROCRYPT 2008, PAPERS.md).  The walk is extract.cuh; this file holds the kernel and its host driver.
#include <cstddef>

#include "batchinv.cuh"
#include "ctx.h"
#include "extract.cuh"

using namespace gs;

namespace gs {

constexpr int GS_EXT_NT = 128;
// resident blocks per SM the kernel is compiled for, by measurement on a B200 (DESIGN.md §4, "Extraction"): G1 3 blocks =
// 168 registers, what it takes unbounded (4 blocks = 128 registers spill and are 1 % slower); G2 3 blocks = 168 registers
// is 14 % faster than unbounded (200 registers, 2 blocks)
#ifndef GS_EXT_G1_BLOCKS
#define GS_EXT_G1_BLOCKS 3
#endif
#ifndef GS_EXT_G2_BLOCKS
#define GS_EXT_G2_BLOCKS 3
#endif

// out[i] = coms[i].1 - a coms[i].0, one thread per commitment, the digits of a in `dg` (the same for every lane)
template <class F>
__global__ void __launch_bounds__(GS_EXT_NT, sizeof(typename F::T) == sizeof(fp) ? GS_EXT_G1_BLOCKS : GS_EXT_G2_BLOCKS)
    k_extract(const Aff<F>* __restrict__ coms, Aff<F>* __restrict__ out, size_t n, extract_digits dg) {
  __shared__ fp sm[2 * GS_EXT_NT];
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool active = i < n;
  Jac<F> acc;
  acc.set_inf();
  if (active) extract_jac<F>(acc, coms[2 * i], coms[2 * i + 1], dg);
  Aff<F> r;
  block_to_affine<GS_EXT_NT>(r, acc, sm);
  if (active) out[i] = r;
}

}  // namespace gs

namespace gsi {

template <class F>
struct ext_side;
template <>
struct ext_side<FpOps> {
  static const g1_aff* key(const crs_dev* c) { return &c->u[0][0]; }
  static bool& valid(gs_ctx* ctx) { return ctx->xkey_valid; }
  static gs_fr& cached(gs_ctx* ctx) { return ctx->xkey; }
  static constexpr const char* bad_key = "extract: xkey is not the extraction key of the loaded CRS (a1 of gs_crs_generate)";
};
template <>
struct ext_side<Fp2Ops> {
  static const g2_aff* key(const crs_dev* c) { return &c->v[0][0]; }
  static bool& valid(gs_ctx* ctx) { return ctx->ykey_valid; }
  static gs_fr& cached(gs_ctx* ctx) { return ctx->ykey; }
  static constexpr const char* bad_key = "extract: ykey is not the extraction key of the loaded CRS (a2 of gs_crs_generate)";
};

template <class F>
static extract_digits digits_of(const gs_fr* key) {
  fr k;
  memcpy(&k, key, sizeof(fr));
  uint32_t c[8];
  fr_from_mont(c, k);
  return make_extract_digits<F>(c);
}

// *all_identity = (coms[i].1 - key coms[i].0 is the identity for every i < n), n device commitments
template <class F>
int extract_all_identity(gs_ctx* ctx, const Aff<F>* coms, size_t n, const gs_fr* key, bool* all_identity) {
  Scratch sc(ctx);
  Aff<F>* dout;
  CUDA_TRY(sc.alloc(&dout, n));
  LAUNCH_CFG((k_extract<F>), n, GS_EXT_NT, 0, coms, dout, n, digits_of<F>(key));
  std::vector<Aff<F>> h(n);
  CUDA_TRY(cudaMemcpyAsync(h.data(), dout, n * sizeof(Aff<F>), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  *all_identity = true;
  for (const Aff<F>& p : h) *all_identity = *all_identity && p.is_inf();
  return GS_OK;
}
template int extract_all_identity<FpOps>(gs_ctx*, const g1_aff*, size_t, const gs_fr*, bool*);
template int extract_all_identity<Fp2Ops>(gs_ctx*, const g2_aff*, size_t, const gs_fr*, bool*);

// The key matches the loaded CRS iff extracting the two key commitments u[0], u[1] (v[0], v[1]) gives the identity
// twice.  Under the hiding key u[1] - iota_1(g1) extracts to -g1, so that key fails as well.  A validated key is
// cached until the next gs_crs_load / gs_crs_generate.
template <class F>
static int key_check(gs_ctx* ctx, const gs_fr* key) {
  if (ext_side<F>::valid(ctx) && memcmp(&ext_side<F>::cached(ctx), key, sizeof(gs_fr)) == 0) return GS_OK;
  bool ok;
  int rc = extract_all_identity<F>(ctx, ext_side<F>::key(ctx->crs), 2, key, &ok);
  if (rc) return rc;
  if (!ok) FAIL(GS_EARG, ext_side<F>::bad_key);
  ext_side<F>::cached(ctx) = *key;
  ext_side<F>::valid(ctx) = true;
  return GS_OK;
}

// out[i] = coms[i].1 - a coms[i].0 for n host commitments.  Batches of more than two chunks are cut into 2^16-element
// chunks that alternate between the context's two streams, as in batch_commit_impl: while the host stages chunk i+1 in
// and chunk i-1 out, the kernel of chunk i runs.
template <class F>
static int extract_side(gs_ctx* ctx, size_t n, const Aff<F>* coms, const extract_digits& dg, Aff<F>* out) {
  const size_t CH = (size_t)1 << 16;
  const size_t step = n > 2 * CH ? CH : n;
  if (step < n && !ctx->stream2) CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
  cudaStream_t main_stream = ctx->stream;
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
    cudaError_t e2 = cudaMemcpyAsync(out + pd.off, pd.dout, pd.cnt * sizeof(Aff<F>), cudaMemcpyDeviceToHost, pd.st);
    if (e2 == cudaSuccess) e2 = cudaStreamSynchronize(pd.st);
    if (ce == cudaSuccess) ce = e2;
    delete pd.sc;
    pd.sc = nullptr;
  };
  size_t idx = 0;
  for (size_t off = 0; off < n && rc == GS_OK && ce == cudaSuccess; off += step, idx++) {
    const size_t cnt = n - off < step ? n - off : step;
    pending_t cur;
    cur.st = (idx & 1) ? ctx->stream2 : main_stream;
    cur.off = off;
    cur.cnt = cnt;
    ctx->stream = cur.st;
    cur.sc = new Scratch(ctx);
    Aff<F>* dcom;
    cudaError_t e2 = upload(ctx, *cur.sc, &dcom, coms + 2 * off, 2 * cnt);
    if (e2 == cudaSuccess) e2 = cur.sc->alloc(&cur.dout, cnt);
    if (e2 != cudaSuccess) {
      ce = e2;
      delete cur.sc;
      break;
    }
    rc = [&]() -> int {
      LAUNCH_CFG((k_extract<F>), cnt, GS_EXT_NT, 0, (const Aff<F>*)dcom, cur.dout, cnt, dg);
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

}  // namespace gsi

using namespace gsi;

extern "C" {

int gs_extract(gs_ctx* ctx, size_t nx, const gs_com1* xcoms, const gs_fr* xkey, size_t ny, const gs_com2* ycoms,
               const gs_fr* ykey, gs_g1* out_x, gs_g2* out_y) {
  if (!ctx) return GS_EARG;
  if (nx && (!xcoms || !xkey || !out_x)) FAIL(GS_EARG, "extract: null pointer on the G1 side");
  if (ny && (!ycoms || !ykey || !out_y)) FAIL(GS_EARG, "extract: null pointer on the G2 side");
  if (!ctx->crs_loaded) FAIL(GS_EARG, "extract: no CRS loaded");
  if (nx == 0 && ny == 0) return GS_OK;
  CUDA_TRY(cudaSetDevice(ctx->device));
  // both keys are checked before anything is written, so a wrong key leaves both outputs untouched
  extract_digits dx, dy;
  int rc;
  if (nx) {
    dx = digits_of<FpOps>(xkey);
    if ((rc = key_check<FpOps>(ctx, xkey))) return rc;
  }
  if (ny) {
    dy = digits_of<Fp2Ops>(ykey);
    if ((rc = key_check<Fp2Ops>(ctx, ykey))) return rc;
  }
  if (nx && (rc = extract_side<FpOps>(ctx, nx, (const g1_aff*)xcoms, dx, (g1_aff*)out_x))) return rc;
  if (ny && (rc = extract_side<Fp2Ops>(ctx, ny, (const g2_aff*)ycoms, dy, (g2_aff*)out_y))) return rc;
  return GS_OK;
}

}  // extern "C"
