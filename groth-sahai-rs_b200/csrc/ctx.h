// Host-side context shared by the translation units of libgs_b200.so (one .cu per kernel family so
// that cicc/ptxas run in parallel; every kernel lives in exactly one TU, device helpers are header
// inline).  Nothing here is part of the C ABI: include/gs_b200.h is.
#pragma once
#include "../../include/gs_b200.h"

#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "shapes.cuh"

// fixed-base window tables of one group (prover_impl.cuh builds them):
//   t[((base*2 + a) * W + w) * H + (d-1)] = d * 2^(c w) * Base.a,  bases u1 u2 W1 (G1) / v1 v2 W2 (G2)
template <class F>
struct gs_fixed_table {
  int c = 0, W = 0;
  size_t H = 0;
  gs::Aff<F>* t = nullptr;
};

struct gs_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t stream2 = nullptr;  // second stream of chunked batches (copy / compute overlap), created on first use
  gs::crs_dev* crs = nullptr;  // device
  bool crs_loaded = false;
  bool xkey_valid = false, ykey_valid = false;  // gs_extract: the last key of each side that matched the loaded CRS
  gs_fr xkey{}, ykey{};                         // (cleared by gs_crs_load / gs_crs_generate)
  gs_fixed_table<gs::FpOps> tab1;
  gs_fixed_table<gs::Fp2Ops> tab2;
  bool crs_lines_valid = false;   // the stored lines and the fixed-base tables are built by the FIRST call that needs them
                                  // (a verify / a commit or prove), not by gs_crs_generate / gs_crs_load
  gs::fp2* crs_lines = nullptr;   // (lambda, mu) per Miller step of the fixed G2 points v1.0 v1.1 v2.0 v2.1 W2.0 W2.1:
                                  // crs_lines[(pid*68 + step)*2 + {0,1}]  (pairing.cu crs_lines_build)
  uint32_t* fe_prog = nullptr;    // op program of the cooperative final exponentiation (finalexp.cu)
  int fe_nops = 0;
  uint64_t launches = 0;
  bool profile = false;
  struct prof_rec {
    const char* name;
    cudaEvent_t e0, e1;
  };
  std::vector<prof_rec> prof;
  size_t verify_batch_max = 23680;  // problems per verify pass (10 waves of k_miller4)
  size_t tile_budget = (size_t)16 << 30;  // bytes of HBM for the evaluated-line tiles of one pairing pass
  size_t split_min = 4736;  // a batch between this size (2 waves of k_miller4) and one pass is still cut in two, one half per
                            // stream, so that partial waves of one half are filled by the other (GS_SPLIT_MIN; 0 = never)
  int lone_walk_jac = 1;    // lone statements walk their G2 points in Jacobian coordinates + one batched inversion
                            // (GS_LONE_WALK_JAC = 0: the affine walk with an inversion per step)
  int pass_streams = 2;   // verify passes of a big batch alternate between this many streams (GS_PASS_STREAMS = 1 | 2)
  int prep_variant = 5;   // resident blocks per SM the line-walk kernel is compiled for (GS_PREP_VARIANT = 4 | 5, experiments)
  size_t rand_pip_min = 4096;   // gs_verify_batch_rand: batches of at least this many proofs sum their pi / theta slots over the
                                // proofs with the bucket method (GS_RAND_PIP_MIN; measured better from 8,192 proofs up: 50.6 vs 51.7 ms)
  size_t pip_min = 2048;  // proof MSMs of one statement with at least this many terms use the bucket method (pippenger.cuh);
  int pip_c = 0;          // measured crossover, DESIGN.md §4.  Overrides for experiments: GS_PIP_MIN, GS_PIP_C (window bits)
  std::string err;
};

#define CUDA_TRY(x)                                               \
  do {                                                            \
    cudaError_t e_ = (x);                                         \
    if (e_ != cudaSuccess) {                                      \
      ctx->err = std::string(#x) + ": " + cudaGetErrorString(e_); \
      return GS_ECUDA;                                            \
    }                                                             \
  } while (0)
#define FAIL(code, msg) \
  do {                  \
    ctx->err = (msg);   \
    return (code);      \
  } while (0)
// launch `kern` with `nthreads` logical threads in blocks of `bs` and `smem` dynamic shared bytes;
// `gy` = gridDim.y (batched kernels: blockIdx.y = instance, see prover.cu)
#define LAUNCH_GRID(kern, nthreads, gy, bs, smem, ...)                    \
  do {                                                                    \
    size_t nt_ = (nthreads);                                              \
    if (nt_ > 0 && (gy) > 0) {                                            \
      dim3 grid_((unsigned)((nt_ + (bs)-1) / (bs)), (unsigned)(gy));      \
      gs_ctx::prof_rec pr_{#kern, nullptr, nullptr};                      \
      if (ctx->profile) {                                                 \
        cudaEventCreate(&pr_.e0);                                         \
        cudaEventCreate(&pr_.e1);                                         \
        cudaEventRecord(pr_.e0, ctx->stream);                             \
      }                                                                   \
      kern<<<grid_, (bs), (smem), ctx->stream>>>(__VA_ARGS__);            \
      if (ctx->profile) {                                                 \
        cudaEventRecord(pr_.e1, ctx->stream);                             \
        ctx->prof.push_back(pr_);                                         \
      }                                                                   \
      ctx->launches++;                                                    \
      CUDA_TRY(cudaGetLastError());                                       \
    }                                                                     \
  } while (0)
#define LAUNCH_CFG(kern, nthreads, bs, smem, ...) LAUNCH_GRID(kern, nthreads, 1, bs, smem, __VA_ARGS__)
#define LAUNCH(kern, nthreads, ...) LAUNCH_GRID(kern, nthreads, 1, 128, 0, __VA_ARGS__)
#define LAUNCH_B(kern, nthreads, nbatch, ...) LAUNCH_GRID(kern, nthreads, nbatch, 128, 0, __VA_ARGS__)

// stream-ordered scratch with RAII release
struct Scratch {
  gs_ctx* ctx;
  cudaStream_t home;  // the stream that was current at construction: everything is released there (stream-ordered), also
                      // when ctx->stream has been switched back by then (passes that alternate between two streams)
  std::vector<void*> ptrs;
  explicit Scratch(gs_ctx* c) : ctx(c), home(c->stream) {}
  template <class T>
  cudaError_t alloc(T** p, size_t count) {
    void* q = nullptr;
    cudaError_t e = cudaMallocAsync(&q, count * sizeof(T) + 16, ctx->stream);
    if (e == cudaSuccess) ptrs.push_back(q);
    *p = (T*)q;
    return e;
  }
  ~Scratch() {
    for (void* q : ptrs) cudaFreeAsync(q, home);
  }
};
// instances per verify pass: verify_batch_max for big batches; half of a medium batch (two streams fill each other's
// partial waves -- the strong-scaling regime of C5: 8,192 proofs per GPU are 3.46 waves of k_miller4); else everything.
// `one_pass`: the caller has already cut the batch into passes (verify_host), no second split inside
static inline size_t verify_pass_size(const gs_ctx* ctx, size_t count, bool shared_x, bool one_pass) {
  if (one_pass) return count;
  if (count > ctx->verify_batch_max) return ctx->verify_batch_max;
  if (ctx->pass_streams == 2 && !ctx->profile && !shared_x && ctx->split_min && count >= ctx->split_min)
    return (((count + 1) / 2) + 31) / 32 * 32;
  return count;
}
// The passes of a big batch, alternating between ctx->stream and the context's second stream.  On every exit path of the
// scope ctx->stream is restored and, once split() has run, ordered after everything queued on the second stream.
struct PassStreams {
  gs_ctx* ctx;
  cudaStream_t s[2];
  bool two = false;
  explicit PassStreams(gs_ctx* c) : ctx(c), s{c->stream, c->stream} {}
  // odd passes run on the second stream (created on first use); with `fork` it first waits for everything queued on the
  // main stream so far (inputs uploaded or produced there)
  cudaError_t split(bool fork) {
    if (!ctx->stream2) {
      cudaError_t e = cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking);
      if (e != cudaSuccess) return e;
    }
    s[1] = ctx->stream2;
    two = true;
    if (!fork) return cudaSuccess;
    cudaEvent_t ev;
    cudaError_t e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming);
    if (e != cudaSuccess) return e;
    cudaEventRecord(ev, s[0]);
    cudaStreamWaitEvent(s[1], ev, 0);
    cudaEventDestroy(ev);
    return cudaSuccess;
  }
  void use(size_t pass) { ctx->stream = s[pass & 1]; }
  ~PassStreams() {
    ctx->stream = s[0];
    if (!two) return;
    cudaEvent_t j;
    if (cudaEventCreateWithFlags(&j, cudaEventDisableTiming) != cudaSuccess) {
      cudaStreamSynchronize(s[1]);
      return;
    }
    cudaEventRecord(j, s[1]);
    cudaStreamWaitEvent(s[0], j, 0);
    cudaEventDestroy(j);
  }
};

template <class T>
static inline cudaError_t upload(gs_ctx* ctx, Scratch& s, T** dst, const void* src, size_t count) {
  cudaError_t e = s.alloc(dst, count);
  if (e != cudaSuccess) return e;
  if (count == 0) return cudaSuccess;
  return cudaMemcpyAsync(*dst, src, count * sizeof(T), cudaMemcpyHostToDevice, ctx->stream);
}

static inline size_t elem_size_A(int type) { return (type == 0 || type == 1) ? sizeof(gs::g1_aff) : sizeof(gs::fr); }
static inline size_t elem_size_B(int type) { return (type == 0 || type == 2) ? sizeof(gs::g2_aff) : sizeof(gs::fr); }
static inline size_t elem_size_T(int type) {
  return type == 0 ? sizeof(gs::fp12) : type == 1 ? sizeof(gs::g1_aff) : type == 2 ? sizeof(gs::g2_aff) : sizeof(gs::fr);
}

// ---- functions that cross translation units (namespace gsi = "internal") ----
namespace gsi {
using namespace gs;

// pairing.cu
int pairing_init(gs_ctx* ctx);  // per-context kernel attributes
int final_exp_init(gs_ctx* ctx);
// X, Y: device slot arrays [2][K][nprob]  ->  ComT values (out_comt, AoS [p][4]) or per-entry verdict
// bytes ok4[4][nprob] (compared with 1 / target).
// With out_partial (AoS [p][4]) the un-exponentiated Miller products are returned instead (sharded statements).
// slot_kind (host, K entries, or null = all GS_SLOT_WALK) tells what is known about Y_k from the shape alone.
constexpr uint8_t GS_SLOT_WALK = 0;     // arbitrary Com2: walk both coordinates
constexpr uint8_t GS_SLOT_WALK_B1 = 1;  // Y_k = (O, y): only coordinate 1 exists (iota_2)
constexpr uint8_t GS_SLOT_FIXED = 2;    // GS_SLOT_FIXED + j: Y_k is the CRS element v_1 (j = 0), v_2 (1) or W2 (2)
constexpr uint8_t GS_SLOT_WALK_SHARED = 0x40;  // arbitrary Com2 that is THE SAME in every problem of the call (the y-commitments of
                                               // a multi-equation statement): walked once when the lines are walked ahead
struct walk_ahead {  // G2 walks started early on the second stream (lone statements), see g2_walk_ahead
  gs_ctx* ctx = nullptr;
  fp2* lines = nullptr;
  uint32_t* dwalk = nullptr;
  int nwalk = 0;
  cudaEvent_t done = nullptr;
  walk_ahead() = default;
  walk_ahead(const walk_ahead&) = delete;
  walk_ahead& operator=(const walk_ahead&) = delete;
  // On EVERY exit (error paths included) the main stream is ordered after the walk before the Scratch that owns the
  // walk's buffers frees them with cudaFreeAsync on the main stream: declare the walk_ahead AFTER that Scratch.
  ~walk_ahead() {
    if (done) {
      if (ctx) cudaStreamWaitEvent(ctx->stream, done, 0);
      cudaEventDestroy(done);
    }
  }
};
int g2_walk_ahead(gs_ctx* ctx, Scratch& sc, const g2_aff* Y, size_t nprob, int K, const uint8_t* slot_kind, walk_ahead* wa);
// Single-entry products with one result PER ACCUMULATOR (gs_verify_each_rand): F[A] = the conjugated Miller value of
// accumulator A (slots [A*S, A*S + S)), neither multiplied over the accumulators nor exponentiated.  The first nf slots of
// every acc_stride-th accumulator (A = 0, acc_stride, 2 acc_stride, ...) are pairs whose G2 side is one of a few points
// shared by the whole call, pts[pid[f]], with lines walked once (lines[(pid*68 + step)*2 + {0: lambda, 1: mu}], g2_lines);
// their Y entries must be the identity so that the per-slot walk skips them.
struct acc_each {
  fp12* F = nullptr;
  int acc_stride = 1;
  int nf = 0;
  int pid[4] = {0, 0, 0, 0};
  const g2_aff* pts = nullptr;
  const fp2* lines = nullptr;
};
int run_pairing_product(gs_ctx* ctx, Scratch& sc, const g1_aff* X, const g2_aff* Y, size_t nprob, int K, fp12* out_comt,
                        uint8_t* ok4, const fp12* target, fp12* out_partial, const uint8_t* slot_kind = nullptr,
                        const walk_ahead* wa = nullptr, int ne = 4, int S_force = 0, const acc_each* each = nullptr);
// lines[(i*68 + step)*2 + {0: lambda, 1: mu}] of the n G2 points pts[i] (device), walked once each; *lines is owned by `sc`
int g2_lines(gs_ctx* ctx, Scratch& sc, const g2_aff* pts, int n, fp2** lines);
int crs_lines_build(gs_ctx* ctx);

// finalexp.cu: f = prod_chunks F[(ch*ne + e)*nprob + p]; g = FE(f); writes out_comt[p*ne+e] and/or ok4[e*nprob + p]
// (ne = 4 entries per problem; ne = 1: single values, `target` then applies to every problem)
int launch_final_exp(gs_ctx* ctx, const fp12* F, size_t nprob, int nchunk, fp12* out_comt, uint8_t* ok4, const fp12* target, int ne = 4);
// finalexp.cu: multiplies groups of chunks together (cooperative kernel) until nchunk <= max_out
int reduce_chunks(gs_ctx* ctx, Scratch& sc, const fp12** F, size_t nprob, int* nchunk, int max_out, int ne = 4);
// finalexp.cu: out[i] = t[i]^(e[i * estride]) for 64-bit exponents, t in the cyclotomic subgroup (GT members are)
int gt_pow64(gs_ctx* ctx, const fp12* t, const uint64_t* e, size_t estride, size_t count, fp12* out);

// prover.cu
int crs_generate_points(gs_ctx* ctx, const gs_g1* p1, const gs_g2* p2, const gs_fr* a1, const gs_fr* a2, const gs_fr* t1,
                        const gs_fr* t2, gs_crs* out);
int crs_derive(gs_ctx* ctx);

// prover_g1.cu / prover_g2.cu (explicit instantiations of prover_impl.cuh)
template <class F>
gs_fixed_table<F>& table_of(gs_ctx* ctx);
template <>
inline gs_fixed_table<FpOps>& table_of<FpOps>(gs_ctx* ctx) { return ctx->tab1; }
template <>
inline gs_fixed_table<Fp2Ops>& table_of<Fp2Ops>(gs_ctx* ctx) { return ctx->tab2; }

template <class F>
int fixed_table_rebuild(gs_ctx* ctx, int c);
template <class F>
void fixed_table_release(gs_ctx* ctx);
template <class F>
int batch_commit_impl(gs_ctx* ctx, size_t n, int base0, int base1, const gs_fr* s0, size_t s0_stride, const gs_fr* s1,
                      size_t s1_stride, size_t nscal, const void* addend, void* out);
// one proof element vector (pi: F = G2, theta: F = G1); `e` = collapsed scalar for scalar-typed sides (else null)
// Batched over `count` proofs (blockIdx.y): per-proof strides are implied by the shapes; `vars_shared` = the
// variable array is one set used by every proof.
template <class F>
int proof_element(gs_ctx* ctx, Scratch& sc, size_t count, int rows, bool group_typed, const fr* sv, const void* dconst,
                  size_t nconst, const void* dvars, size_t nvars, bool vars_shared, int ncoef, const fr* coef, size_t coef_rs,
                  const fr* e, Aff<F>* dout);
// rerandomisation of committed proofs (prover.cu gs_rerandomize_batch): c' = c + R' key for n commitments, and one
// rerandomised proof element vector per proof (sv / rg: the scalar rows, see prover_impl.cuh)
template <class F>
int rerand_commit(gs_ctx* ctx, size_t n, int ns, const fr* dR, const Aff<F>* dcom, Aff<F>* dout);
template <class F>
int rerand_element(gs_ctx* ctx, Scratch& sc, size_t count, int rows, bool group_typed, const fr* sv, const fr* rg,
                   const void* dconst, size_t nconst, const Aff<F>* dcom, size_t ncom, bool coms_shared, int ncoef,
                   const fr* coef, const fr* e, const Aff<F>* dold, Aff<F>* dout);
template <class F>
int com_matmul_impl(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* lhs, const void* mat, void* out);

}  // namespace gsi
