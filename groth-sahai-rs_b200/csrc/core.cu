// libgs_b200.so -- C ABI over the sm_100a kernels (include/gs_b200.h): context, measurement hooks, CRS.
// No CPU fallback anywhere: every entry point launches CUDA kernels or fails with GS_ECUDA.
#include "ctx.h"

#include <cstdlib>

using namespace gs;

static_assert(sizeof(gs_fr) == sizeof(fr), "fr layout");
static_assert(sizeof(gs_g1) == sizeof(g1_aff), "g1 layout");
static_assert(sizeof(gs_g2) == sizeof(g2_aff), "g2 layout");
static_assert(sizeof(gs_gt) == sizeof(fp12), "gt layout");
static_assert(sizeof(gs_com1) == 2 * sizeof(g1_aff), "com1 layout");
static_assert(sizeof(gs_com2) == 2 * sizeof(g2_aff), "com2 layout");

namespace gsi {
extern template void fixed_table_release<FpOps>(gs_ctx*);
extern template void fixed_table_release<Fp2Ops>(gs_ctx*);
extern template int fixed_table_rebuild<FpOps>(gs_ctx*, int);
extern template int fixed_table_rebuild<Fp2Ops>(gs_ctx*, int);
}  // namespace gsi

extern "C" {

int gs_ctx_create(int device, gs_ctx** out) {
  if (!out) return GS_EARG;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || device < 0 || device >= ndev) return GS_ECUDA;
  gs_ctx* ctx = new gs_ctx();
  ctx->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaMalloc(&ctx->crs, sizeof(crs_dev)) != cudaSuccess) {
    delete ctx;
    return GS_ECUDA;
  }
  // keep freed scratch in the pool instead of returning it to the driver after every call
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t thr = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
  }
  if (const char* e = getenv("GS_PIP_MIN")) ctx->pip_min = (size_t)strtoull(e, nullptr, 10);
  if (const char* e = getenv("GS_PIP_C")) ctx->pip_c = atoi(e);
  if (const char* e = getenv("GS_RAND_PIP_MIN")) ctx->rand_pip_min = (size_t)strtoull(e, nullptr, 10);
  if (const char* e = getenv("GS_PREP_VARIANT")) ctx->prep_variant = atoi(e);
  if (const char* e = getenv("GS_PASS_STREAMS")) ctx->pass_streams = atoi(e);
  if (const char* e = getenv("GS_LONE_WALK_JAC")) ctx->lone_walk_jac = atoi(e);
  if (const char* e = getenv("GS_SPLIT_MIN")) ctx->split_min = (size_t)strtoull(e, nullptr, 10);
  if (const char* e = getenv("GS_VERIFY_BATCH_MAX")) {  // problems per verify pass (tests: several passes on a small batch)
    const size_t v = (size_t)strtoull(e, nullptr, 10);
    if (v >= 1) ctx->verify_batch_max = v;
  }
  // deep call chains (Fp12 -> Fp6 -> Fp2) with big local frames
  cudaDeviceSetLimit(cudaLimitStackSize, 32 * 1024);
  if (gsi::pairing_init(ctx) != GS_OK || gsi::final_exp_init(ctx) != GS_OK) {
    delete ctx;
    return GS_ECUDA;
  }
  *out = ctx;
  return GS_OK;
}

void gs_ctx_destroy(gs_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  gsi::fixed_table_release<FpOps>(ctx);
  gsi::fixed_table_release<Fp2Ops>(ctx);
  if (ctx->crs_lines) cudaFree(ctx->crs_lines);
  if (ctx->fe_prog) cudaFree(ctx->fe_prog);
  cudaFree(ctx->crs);
  if (ctx->stream2) cudaStreamDestroy(ctx->stream2);
  cudaStreamDestroy(ctx->stream);
  delete ctx;
}

const char* gs_last_error(const gs_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }
uint64_t gs_launch_count(const gs_ctx* ctx) { return ctx ? ctx->launches : 0; }
void* gs_stream(const gs_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }


int gs_profile_enable(gs_ctx* ctx, int on) {
  if (!ctx) return GS_EARG;
  ctx->profile = on != 0;
  return GS_OK;
}

int gs_profile_read(gs_ctx* ctx, char* buf, size_t cap) {
  if (!ctx || !buf || cap == 0) return -GS_EARG;
  cudaSetDevice(ctx->device);
  if (cudaStreamSynchronize(ctx->stream) != cudaSuccess) return -GS_ECUDA;
  std::vector<std::string> names;
  std::vector<double> ms;
  std::vector<int> cnt;
  for (auto& r : ctx->prof) {
    float t = 0;
    cudaEventElapsedTime(&t, r.e0, r.e1);
    cudaEventDestroy(r.e0);
    cudaEventDestroy(r.e1);
    size_t i = 0;
    for (; i < names.size(); i++)
      if (names[i] == r.name) break;
    if (i == names.size()) {
      names.push_back(r.name);
      ms.push_back(0);
      cnt.push_back(0);
    }
    ms[i] += t;
    cnt[i]++;
  }
  ctx->prof.clear();
  std::string out;
  for (size_t i = 0; i < names.size(); i++) {
    char line[256];
    snprintf(line, sizeof line, "%s %d %.6f\n", names[i].c_str(), cnt[i], ms[i]);
    out += line;
  }
  size_t n = out.size() < cap - 1 ? out.size() : cap - 1;
  memcpy(buf, out.data(), n);
  buf[n] = 0;
  return (int)n;
}

}  // extern "C"

// register-only Fp product chain (the measured integer-multiply roofline)
__global__ void __launch_bounds__(256) k_diag_fpmul(fp* out, const fp* in, int iters) {
  int t = blockIdx.x * blockDim.x + threadIdx.x;
  fp x = in[t], y = in[t + 1];
  for (int i = 0; i < iters; i++) fp::mul(x, x, y);
  out[t] = x;
}

extern "C" int gs_diag_fpmul_rate(gs_ctx* ctx, double* fpmul_per_sec) {
  if (!ctx || !fpmul_per_sec) return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, ctx->device));
  const int blocks = prop.multiProcessorCount * 2, threads = 256, iters = 4000;
  Scratch sc(ctx);
  fp *in, *out;
  CUDA_TRY(sc.alloc(&in, (size_t)blocks * threads + 1));
  CUDA_TRY(sc.alloc(&out, (size_t)blocks * threads));
  CUDA_TRY(cudaMemsetAsync(in, 1, ((size_t)blocks * threads + 1) * sizeof(fp), ctx->stream));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  double best = 0;
  for (int rep = 0; rep < 4; rep++) {
    cudaEventRecord(e0, ctx->stream);
    k_diag_fpmul<<<blocks, threads, 0, ctx->stream>>>(out, in, iters);
    cudaEventRecord(e1, ctx->stream);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    double rate = (double)blocks * threads * iters / (ms * 1e-3);
    if (rep > 0 && rate > best) best = rate;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  *fpmul_per_sec = best;
  return GS_OK;
}


static int load_crs_device(gs_ctx* ctx, const gs_crs* crs) {
  ctx->xkey_valid = ctx->ykey_valid = false;  // gs_extract checked its cached keys against the previous CRS
  ctx->tkey_valid = false;                      // gs_simulate likewise
  crs_dev h;
  memset(&h, 0, sizeof(h));
  for (int k = 0; k < 2; k++)
    for (int a = 0; a < 2; a++) {
      memcpy(&h.u[k][a], &crs->u[k].p[a], sizeof(g1_aff));
      memcpy(&h.v[k][a], &crs->v[k].p[a], sizeof(g2_aff));
    }
  memcpy(&h.g1, &crs->g1_gen, sizeof(g1_aff));
  memcpy(&h.g2, &crs->g2_gen, sizeof(g2_aff));
  CUDA_TRY(cudaMemcpyAsync(ctx->crs, &h, sizeof(h), cudaMemcpyHostToDevice, ctx->stream));
  int rc = gsi::crs_derive(ctx);
  if (rc) return rc;
  // Everything derived from the key that only SOME calls need is built by the first call that needs it: the fixed-base
  // window tables of u, v, W (first commit / prove: batch_commit_impl, proof_element) and the stored Miller lines of
  // v1, v2, W2 (first verify: crs_lines_build).  generate_crs itself is 6 scalar multiplications and one pairing in the
  // reference (generator.rs:81-118); the 17 ms of table builds that used to sit here made it ~15x slower than the CPU.
  gsi::fixed_table_release<FpOps>(ctx);
  gsi::fixed_table_release<Fp2Ops>(ctx);
  ctx->crs_lines_valid = false;
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  ctx->crs_loaded = true;
  return GS_OK;
}

extern "C" {

int gs_crs_load(gs_ctx* ctx, const gs_crs* crs) {
  if (!ctx || !crs) return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  return load_crs_device(ctx, crs);
}

int gs_crs_generate(gs_ctx* ctx, const gs_g1* p1, const gs_g2* p2, const gs_fr* a1, const gs_fr* a2, const gs_fr* t1,
                    const gs_fr* t2, gs_crs* out) {
  if (!ctx || !p1 || !p2 || !a1 || !a2 || !t1 || !t2 || !out) return GS_EARG;
  CUDA_TRY(cudaSetDevice(ctx->device));
  int rc = gsi::crs_generate_points(ctx, p1, p2, a1, a2, t1, t2, out);
  if (rc) return rc;
  rc = gs_pairing(ctx, 1, p1, p2, &out->gt_gen);  // generator.rs:116
  if (rc) return rc;
  return load_crs_device(ctx, out);
}

}  // extern "C"
