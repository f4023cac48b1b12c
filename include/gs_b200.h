/* gs_b200.h -- C ABI of the B200-native Groth-Sahai engine (libgs_b200.so).
 *
 * The reference (jdwhite48/groth-sahai-rs) has no FFI layer: its boundary is its public
 * Rust API (SURVEY.md §8b).  These entry points are what a thin Rust shim for the hot path
 * binds (see INTEGRATION.md for the `extern "C"` block and the shim); each one names the
 * reference function it replaces (paths relative to /root/reference).
 *
 * Data layout (identical to arkworks' in-memory representation, so the shim passes slices
 * without conversion):
 *   Fr   : 4 x u64 little-endian limbs, Montgomery form, R = 2^256            (32 B)
 *   Fp   : 6 x u64 little-endian limbs, Montgomery form, R = 2^384            (48 B)
 *   G1   : affine x || y                                                      (96 B)
 *   G2   : affine x.c0 || x.c1 || y.c0 || y.c1                                (192 B)
 *          the point at infinity is encoded as all-zero bytes (not on either curve)
 *   Com1 : two G1 (192 B)      Com2 : two G2 (384 B)
 *   GT   : Fp12 = 12 Fp in tower order c0.c0.c0, c0.c0.c1, c0.c1.c0, ...      (576 B)
 *   ComT : four GT, row-major [e(x0,y0), e(x0,y1), e(x1,y0), e(x1,y1)]        (2304 B)
 *   Matrix<Fr> : dense row-major.
 *
 * Group elements must lie in the order-r subgroups (what arkworks' validated deserialisation guarantees for
 * every G1Affine / G2Affine; gs_g1_decompress / gs_g2_decompress check it): the kernels use the curve
 * endomorphisms, which act as scalars only there.
 *
 * All pointers are HOST pointers unless the function name ends in `_dev`.  Randomness is
 * always supplied by the caller, drawn in the reference's order (commit.rs:85-88,
 * prove.rs:123-126), which is what makes results bit-reproducible.
 *
 * Every function returns GS_OK or an error code; gs_last_error() gives the message.  The
 * reference signals the same conditions by assert!/panic; the shim re-panics on GS_EDIM.
 * There is no CPU fallback: without a CUDA device gs_ctx_create fails with GS_ECUDA.
 */
#ifndef GS_B200_H
#define GS_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GS_OK 0
#define GS_EDIM 1   /* dimension / argument error (reference: assert_eq! panic) */
#define GS_ECUDA 2  /* CUDA runtime error */
#define GS_EARG 3   /* null pointer / bad enum */

/* EquType byte, src/statement.rs:68-73 */
#define GS_PPE 0
#define GS_MSMEG1 1
#define GS_MSMEG2 2
#define GS_QUAD 3

typedef struct gs_ctx gs_ctx;

typedef struct { uint64_t l[4]; } gs_fr;
typedef struct { uint64_t x[6], y[6]; } gs_g1;
typedef struct { uint64_t x[12], y[12]; } gs_g2;
typedef struct { gs_g1 p[2]; } gs_com1;
typedef struct { gs_g2 p[2]; } gs_com2;
typedef struct { uint64_t c[72]; } gs_gt;
typedef struct { gs_gt e[4]; } gs_comt;

/* CRS<E>, src/generator.rs:36-42 (u, v, g1_gen, g2_gen, gt_gen) */
typedef struct {
  gs_com1 u[2];
  gs_com2 v[2];
  gs_g1 g1_gen;
  gs_g2 g2_gen;
  gs_gt gt_gen;
} gs_crs;

/* ---- context ------------------------------------------------------------------------- */
/* One context per host thread and per GPU (owns a stream, the device copy of the CRS, the
 * fixed-base tables and scratch).  `device` is the CUDA ordinal. */
int gs_ctx_create(int device, gs_ctx** out);
void gs_ctx_destroy(gs_ctx* ctx);
const char* gs_last_error(const gs_ctx* ctx);
/* number of CUDA kernels this context has launched so far (bench.py's gpu_launches) */
uint64_t gs_launch_count(const gs_ctx* ctx);
/* the cudaStream_t the context launches on (as an opaque pointer, for event timing) */
void* gs_stream(const gs_ctx* ctx);

/* ---- measurement hooks (bench.py) -------------------------------------------------------- */
/* When enabled, every kernel launch is bracketed by CUDA events on gs_stream(). */
int gs_profile_enable(gs_ctx* ctx, int on);
/* Synchronises, then writes one line per kernel: "<name> <launches> <total_ms>\n" (and clears the log).
 * Returns the number of bytes written (truncated to cap-1) or a negative error code. */
int gs_profile_read(gs_ctx* ctx, char* buf, size_t cap);
/* Register-only Fp Montgomery-product chain on every SM: the measured integer-multiply roofline,
 * in Fp products per second (1 product = 600 IMAD-equivalents in SURVEY.md §8d's accounting). */
int gs_diag_fpmul_rate(gs_ctx* ctx, double* fpmul_per_sec);

/* ---- CRS ------------------------------------------------------------------------------ */
/* CRS::generate_crs, src/generator.rs:81-118.  The six values are the reference's RNG draws
 * in its order (p1 <- G1, p2 <- G2, a1, a2, t1, t2 <- Fr, :86-93).  Also loads the result. */
int gs_crs_generate(gs_ctx* ctx, const gs_g1* p1, const gs_g2* p2, const gs_fr* a1, const gs_fr* a2,
                    const gs_fr* t1, const gs_fr* t2, gs_crs* out);
/* Makes `crs` the context's key (any `&CRS<E>` argument of the reference): uploads it and
 * builds the fixed-base window tables for u1, u2, W1 = u2 + (O, g1) and v1, v2, W2. */
int gs_crs_load(gs_ctx* ctx, const gs_crs* crs);

/* ---- commitments (src/prover/commit.rs) ----------------------------------------------- */
/* batch_commit_G1 :78-100 -- c_i = iota_1(X_i) + R[i][0] u1 + R[i][1] u2;  rand is n x 2 */
int gs_batch_commit_g1(gs_ctx* ctx, size_t n, const gs_g1* xvars, const gs_fr* rand, gs_com1* out);
/* batch_commit_G2 :178-200 */
int gs_batch_commit_g2(gs_ctx* ctx, size_t n, const gs_g2* yvars, const gs_fr* rand, gs_com2* out);
/* batch_commit_scalar_to_B1 :125-156 -- c_i = x_i W1 + r_i u1;  rand is n x 1 */
int gs_batch_commit_scalar_b1(gs_ctx* ctx, size_t n, const gs_fr* xs, const gs_fr* rand, gs_com1* out);
/* batch_commit_scalar_to_B2 :225-256 */
int gs_batch_commit_scalar_b2(gs_ctx* ctx, size_t n, const gs_fr* ys, const gs_fr* rand, gs_com2* out);

/* ---- proofs (src/prover/prove.rs) ------------------------------------------------------ */
/* Provable::prove for the four equation types (:92-171, :195-274, :298-379, :409-488).
 * m x-variables, n y-variables, gamma is m x n.  Variables / constants are G1 / G2 points or
 * Fr scalars depending on `type` (see SURVEY.md §3.6):
 *   a_consts : n elements (G1 for PPE, MSMEG1; Fr otherwise)     b_consts : m (G2 for PPE, MSMEG2)
 *   xvars    : m elements (G1 for PPE, MSMEG1; Fr otherwise)     yvars    : n (G2 for PPE, MSMEG2)
 *   x_rand   : m x cx  (cx = 2 for G1 variables, 1 for scalars)   y_rand : n x cy
 *   pf_rand  : T, cy x cx row-major (the reference's draw order)
 *   out_pi   : cx Com2      out_theta : cy Com1 */
int gs_prove(gs_ctx* ctx, int type, size_t m, size_t n, const void* a_consts, const void* b_consts,
             const gs_fr* gamma, const void* xvars, const void* yvars, const gs_fr* x_rand,
             const gs_fr* y_rand, const gs_fr* pf_rand, gs_com2* out_pi, gs_com1* out_theta);

/* `count` independent Provable::prove calls of one type and shape in one pass (the reference proves equation
 * by equation, prove.rs:92-171; a statement with many equations -- BASELINE.json configs[3] -- is a batch of
 * those).  Per-proof arrays are contiguous as in gs_verify_batch: a_consts[count][n], b_consts[count][m],
 * gamma[count][m][n], pf_rand[count][cy][cx]; with shared_vars != 0 the witnesses and their commitment
 * randomness (xvars, yvars, x_rand, y_rand) are ONE set used by every equation, otherwise [count][...].
 * out_pi[count][cx], out_theta[count][cy].  Results are identical to `count` gs_prove calls. */
int gs_prove_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                   const void* b_consts, const gs_fr* gamma, const void* xvars, const void* yvars,
                   const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, int shared_vars,
                   gs_com2* out_pi, gs_com1* out_theta);

/* ---- rerandomisation of committed proofs (not in the reference) ---------------------------------- */
/* Turns a CProof (commitments + proof) into a fresh-looking one for the same statement without the witnesses or the
 * old randomness (Belenkiy et al., CRYPTO 2009; PAPERS.md).  With fresh R' = x_rand (m x cx), S' = y_rand (n x cy)
 * and T' = pf_rand (cy x cx, as for gs_prove):
 *   c' = c + R' u_x                     d' = d + S' v_y
 *   pi'    = pi    + R'^T iota_y(B) + (R'^T Gamma) d + (R'^T Gamma S' - T'^T) v_y
 *   theta' = theta + S'^T iota_x(A) + (S'^T Gamma^T) c + T' u_x
 * (u_x = u[..cx], v_y = v[..cy]; iota = iota_1/2 on a group-typed side, x W1 / y W2 on a scalar-typed one).  The
 * result is byte for byte commit + prove of the same witnesses under R + R', S + S', T + T' + S'^T Gamma^T R: with
 * uniform R', S', T' it is distributed exactly as a fresh proof.  Arrays as gs_prove_batch / gs_verify_batch:
 * a_consts[count][n], b_consts[count][m], gamma[count][m][n], pi[count][cx], theta[count][cy], pf_rand[count][cy][cx],
 * out_pi[count][cx], out_theta[count][cy]; xcoms, ycoms, x_rand, y_rand, out_xcoms, out_ycoms are [count][...], or ONE
 * set used by every equation when shared_coms != 0 (a multi-equation statement over one set of commitments).
 * Return codes as gs_prove_batch.  gs_rerandomize is the batch of one. */
int gs_rerandomize(gs_ctx* ctx, int type, size_t m, size_t n, const void* a_consts, const void* b_consts,
                   const gs_fr* gamma, const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                   const gs_com1* theta, const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand,
                   gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta);
int gs_rerandomize_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                         const void* b_consts, const gs_fr* gamma, const gs_com1* xcoms, const gs_com2* ycoms,
                         const gs_com2* pi, const gs_com1* theta, const gs_fr* x_rand, const gs_fr* y_rand,
                         const gs_fr* pf_rand, int shared_coms, gs_com1* out_xcoms, gs_com2* out_ycoms,
                         gs_com2* out_pi, gs_com1* out_theta);

/* ---- extraction with the binding key (not in the reference) ------------------------------------ */
/* Opens commitments with the binding key's trapdoor (Groth & Sahai, EUROCRYPT 2008; PAPERS.md).
 * X_i = xcoms[i].1 - xkey * xcoms[i].0 (G1), Y_i = ycoms[i].1 - ykey * ycoms[i].0 (G2); xkey = a1, ykey = a2 of
 * gs_crs_generate.  Commitments of scalars give x*g1 / y*g2.  Either side may be empty (n = 0: its pointers may be null).
 * A key is accepted iff it opens the loaded key's own commitments u[0], u[1] (v[0], v[1]) to the identity; otherwise, and
 * under a hiding CRS, GS_EARG with nothing written.  GS_EARG as well without a loaded CRS or for a null pointer on a
 * non-empty side. */
int gs_extract(gs_ctx* ctx, size_t nx, const gs_com1* xcoms, const gs_fr* xkey, size_t ny, const gs_com2* ycoms,
               const gs_fr* ykey, gs_g1* out_x, gs_g2* out_y);

/* ---- zero-knowledge simulation with the hiding key (not in the reference) ------------------------ */
/* Makes accepting proofs WITHOUT witnesses with the hiding key's trapdoor (Groth & Sahai, EUROCRYPT 2008; PAPERS.md).
 * Whoever holds tkey = (t1, t2) of a hiding CRS can make proofs that verify under that CRS for ANY MSMEG1, MSMEG2 or Quad
 * statement and any PPE statement with target 1, true or not; they are distributed exactly like real proofs.  Under the
 * hiding key W1 = u[1] + iota_1(g1) = t1 u[0] and W2 = t2 v[0].  With R = x_rand (m x cx), S = y_rand (n x cy) and
 * T = pf_rand (cy x cx), drawn as for commit + prove:
 *   c = R u_x                         d = S v_y                     (commitments of O / 0)
 *   pi    = R^T iota_y(B) + (R^T Gamma S - T^T) v_y  [- t1 iota_2(T2)   MSMEG2]
 *   theta = S^T iota_x(A) + T u_x                    [- t2 iota_1(T1)   MSMEG1;   - t t2 W1   Quad]
 * i.e. the prover with every witness O / 0 and the target absorbed through the trapdoor.  Arrays as gs_rerandomize_batch
 * (target[count] as gs_verify_batch); with shared_coms != 0, x_rand, y_rand, out_xcoms and out_ycoms are ONE set for every
 * equation.  Return codes as gs_prove_batch, and GS_EARG, with nothing written, when tkey is not the loaded CRS's
 * simulation key (every binding CRS fails), for a PPE target other than 1, without a loaded CRS, or for a null pointer.
 * count == 0 returns GS_OK.  gs_simulate is the batch of one. */
int gs_simulate(gs_ctx* ctx, int type, size_t m, size_t n, const void* a_consts, const void* b_consts,
                const gs_fr* gamma, const void* target, const gs_fr* x_rand, const gs_fr* y_rand,
                const gs_fr* pf_rand, const gs_fr* tkey /* [2] = t1, t2 */, gs_com1* out_xcoms,
                gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta);
int gs_simulate_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                      const void* b_consts, const gs_fr* gamma, const void* target, const gs_fr* x_rand,
                      const gs_fr* y_rand, const gs_fr* pf_rand, int shared_coms, const gs_fr* tkey,
                      gs_com1* out_xcoms, gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta);

/* ---- zero knowledge for PPE targets (not in the reference) ---------------------------------------- */
/* gs_simulate_batch takes PPE statements with target 1 only.  A PPE with a target given as K >= 1 public pairs,
 *     sum_j e(A_j, Y_j) + sum_i e(X_i, B_i) + sum_ij gamma_ij e(X_i, Y_j) = sum_k e(P_k, Q_k),
 * is proved zero-knowledge as the augmented statement of Groth & Sahai (EUROCRYPT 2008; PAPERS.md):
 *   PPE'  target 1, x-variables (X_1..X_m, Z_1..Z_K), b' = (B_1..B_m, -Q_1..-Q_K), a' = A, Gamma' = Gamma + K zero rows;
 *   L_k   (k = 1..K) the MSMEG1 equation Z_k - delta P_k = O: x-variable Z_k, scalar y-variable delta, a = [-P_k],
 *         b = [1], Gamma = [[0]], target O.  The x-commitment of L_k is c_{m+k} of PPE'.
 * delta's commitment is FIXED: W2 = 1 W2 + 0 v[0], which the verifier takes from the loaded CRS, never from the proof.
 * Under a binding CRS it binds delta = 1, so Z_k = P_k and PPE' is the original equation.  Under a hiding CRS
 * W2 = t2 v[0] is also the commitment of 0 with randomness t2: the simulator proves L_k with Z_k = O, delta = 0.
 *   prove    witness (X, Y, Z = P, delta = 1): c = commit(X | P) under R, d = commit(Y) under S (gs_batch_commit_g1 / _g2),
 *            PPE' proved under T (gs_prove_batch), L_k proved with xvars [P_k], yvars [1], x_rand = row m+k of R,
 *            y_rand [0] and T_k (gs_prove_batch of MSMEG1).
 *   simulate c = R u, d = S v (commitments of O), PPE' simulated with target 1 (gs_simulate_batch), L_k simulated as
 *            MSMEG1 with target O, x_rand = row m+k of R, y_rand [t2] and T_k.
 *   verify   accepted iff PPE' verifies on (c, d, pi, theta) and every L_k on ([c_{m+k}], [W2], lin_pi_k, lin_theta_k).
 * Real and simulated proofs are honest proofs of the same augmented statement, identically distributed under a hiding
 * CRS.  Arrays are proof-major (count statements of one shape m, n, K):
 *   a_consts[count][n] (G1), b_consts[count][m] (G2), gamma[count][m][n], tp[count][K] (G1), tq[count][K] (G2),
 *   xvars[count][m], yvars[count][n], x_rand[count][m+K][2], y_rand[count][n][2], pf_rand[count][2][2],
 *   lin_rand[count][K][1][2]; out_xcoms[count][m+K], out_ycoms[count][n], out_pi[count][2], out_theta[count][2],
 *   out_lin_pi[count][K][2], out_lin_theta[count][K][1] (verify reads the same names without out_).
 * The simulator takes no witnesses and the hiding key tkey = (t1, t2), checked as for gs_simulate_batch.
 * GS_EDIM for m, n or K = 0 (a target-1 PPE needs no augmented statement: gs_prove / gs_simulate) or m + K, n over 2^20;
 * GS_EARG, with nothing written, for a null pointer, no loaded CRS, or a tkey that is not the loaded CRS's simulation key
 * (every binding CRS fails).  count == 0 returns GS_OK.  out_ok[i] = 1 iff statement i verifies. */
int gs_zk_ppe_prove_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                          const gs_g2* b_consts, const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq,
                          const gs_g1* xvars, const gs_g2* yvars, const gs_fr* x_rand, const gs_fr* y_rand,
                          const gs_fr* pf_rand, const gs_fr* lin_rand, gs_com1* out_xcoms, gs_com2* out_ycoms,
                          gs_com2* out_pi, gs_com1* out_theta, gs_com2* out_lin_pi, gs_com1* out_lin_theta);
int gs_zk_ppe_simulate_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                             const gs_g2* b_consts, const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq,
                             const gs_fr* x_rand, const gs_fr* y_rand, const gs_fr* pf_rand, const gs_fr* lin_rand,
                             const gs_fr* tkey /* [2] = t1, t2 */, gs_com1* out_xcoms, gs_com2* out_ycoms,
                             gs_com2* out_pi, gs_com1* out_theta, gs_com2* out_lin_pi, gs_com1* out_lin_theta);
/* Rerandomisation of zero-knowledge PPE proofs without the witness (Belenkiy et al., CRYPTO 2009; PAPERS.md): whoever
 * holds a proof of the statements above -- real or simulated -- turns it into a fresh-looking proof of the same statement.
 * With fresh R' = x_rand[count][m+K][2], S' = y_rand[count][n][2], T' = pf_rand[count][2][2] and T'_k =
 * lin_rand[count][K][1][2] (the layouts of gs_zk_ppe_prove_batch):
 *   PPE'  gs_rerandomize_batch of the augmented statement (b' = B | -Q, Gamma' = Gamma + K zero rows) under R', S', T';
 *         this moves c_{m+k}, the x-commitment L_k shares, by row m+k of R'.
 *   L_k   delta's fresh randomness is 0 (its commitment stays W2, which the verifier takes from the CRS), so with
 *         Gamma = 0 and b = [1] only fixed-base terms remain:
 *           lin_pi'_c  = lin_pi_c + R'[m+k][c] W2 - T'_k[c] v[0]   (c = 0, 1)
 *           lin_theta' = lin_theta + T'_k[0] u[0] + T'_k[1] u[1]
 * P_k is multiplied by delta's fresh randomness only, so tp is not an argument.  The output is byte for byte what
 * gs_zk_ppe_prove_batch of the same witnesses makes under R + R', S + S', T + T' + S'^T Gamma'^T R and T_k + T'_k; for a
 * simulated input, what gs_zk_ppe_simulate_batch makes under the same combined randomness (delta's randomness still t2).
 * With uniform fresh randomness the output is distributed exactly as a fresh zk proof, so real and simulated proofs stay
 * indistinguishable.  Rerandomisation does NOT validate its input: a proof that fails verification still fails
 * afterwards (the verification error is unchanged).  No trapdoor is needed; binding and hiding CRSs alike.  Arrays and
 * return codes as gs_zk_ppe_prove_batch (inputs under the verify names, outputs under out_); count == 0 returns GS_OK
 * and writes nothing. */
int gs_zk_ppe_rerandomize_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                                const gs_g2* b_consts, const gs_fr* gamma, const gs_g2* tq, const gs_com1* xcoms,
                                const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const gs_com2* lin_pi,
                                const gs_com1* lin_theta, const gs_fr* x_rand, const gs_fr* y_rand,
                                const gs_fr* pf_rand, const gs_fr* lin_rand, gs_com1* out_xcoms,
                                gs_com2* out_ycoms, gs_com2* out_pi, gs_com1* out_theta, gs_com2* out_lin_pi,
                                gs_com1* out_lin_theta);
int gs_zk_ppe_verify_batch(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                           const gs_g2* b_consts, const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq,
                           const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta,
                           const gs_com2* lin_pi, const gs_com1* lin_theta, uint8_t* out_ok);
/* Randomised PER-STATEMENT verification of the same statements, an opt-in like gs_verify_each_rand: out_ok[i] = 1 iff
 * statement i verifies, except with probability <= 2^-62 over `rho` for every bad statement on its own.  All 1 + K
 * equations of statement i have target 1 (PPE' by construction, L_k with target O).  Every equation e gets weights of its
 * own, (sigma_e, tau_e) = the low 63 bits of two words of rho, and the call one beta from a whole 64-bit word:
 *   PPE' of statement i:  rho[2i], rho[2i + 1];
 *   L_k of statement i:   rho[2 count + 2(iK + k)], rho[2 count + 2(iK + k) + 1];
 *   beta:                 rho[2 count (1 + K)]            (rho has 2 count (1 + K) + 1 words).
 * Each equation's slots are folded as gs_verify_each_rand folds them, and statement i is accepted iff
 *     FE( prod over e in {PPE', L_1..L_K} of prod_k e( sigma_e X_k.0 + tau_e X_k.1 ,  beta Y_k.0 + Y_k.1 ) ) == 1
 * -- one folded pairing product and ONE final exponentiation per statement, however large K is (csrc/verify.cu,
 * "randomised per-statement verification of zk PPEs").  L_k's y-commitment is W2 of the loaded CRS, never an input.  A
 * statement the exact check rejects passes only if a non-zero polynomial of degree 2 in the weights vanishes.  Arrays as
 * for gs_zk_ppe_verify_batch; GS_EDIM for m, n or K = 0 or too many variables, GS_EARG for a null pointer (rho included)
 * or no loaded CRS; count == 0 returns GS_OK and writes nothing.  An all-zero rho accepts everything (the check is then
 * vacuous).  The verdicts are not bit-comparable with gs_zk_ppe_verify_batch's. */
int gs_zk_ppe_verify_each_rand(gs_ctx* ctx, size_t count, size_t m, size_t n, size_t K, const gs_g1* a_consts,
                               const gs_g2* b_consts, const gs_fr* gamma, const gs_g1* tp, const gs_g2* tq,
                               const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta,
                               const gs_com2* lin_pi, const gs_com1* lin_theta, const uint64_t* rho, uint8_t* out_ok);

/* ---- verification (src/verifier.rs)----------------------------------------------------- */
/* Verifiable::verify :23-157 for `count` independent (equation, proof) instances of the same
 * type and shape, each laid out contiguously with the given element counts:
 *   a_consts[count][n], b_consts[count][m], gamma[count][m][n], target[count],
 *   xcoms[count][m], ycoms[count][n], pi[count][cx], theta[count][cy].
 * target is GT (PPE), G1 (MSMEG1), G2 (MSMEG2) or Fr (Quad).  out_ok[i] = 1 iff lhs == rhs. */
int gs_verify_batch(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                    const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                    const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, uint8_t* out_ok);
/* Same with DEVICE pointers (inputs already resident in HBM), asynchronous on gs_stream();
 * out_ok_dev is a device buffer of `count` bytes. */
int gs_verify_batch_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                        const void* b_consts, const gs_fr* gamma, const void* target,
                        const gs_com1* xcoms, const gs_com2* ycoms, const gs_com2* pi,
                        const gs_com1* theta, uint8_t* out_ok_dev);

/* ---- one large statement sharded over several GPUs (SURVEY.md §8e) --------------------------- */
/* Verifiable::verify :23-157 split by SLOT: the pairing-product equation of a statement is a product of
 * K = n + (m or 1) + cx + cy (+1) Miller pairs per ComT entry; rank `rank` of `world` owns the slots
 * k = rank (mod world), evaluates the statement MSM only for those (columns of Gamma) and returns the
 * UN-exponentiated Miller products out_partial[count][4].  Inputs are the FULL arrays of gs_verify_batch
 * on every rank.  The ranks exchange their 4 x 576 B per statement (one all-gather) and any of them
 * finishes with gs_verify_finish.  The reference has no distributed mode; this replaces its Rayon
 * parallelism over left_mul outputs (src/data_structures.rs:657-728) for statements too big for one GPU's
 * latency budget.  rank 0 of world 1 followed by gs_verify_finish(nparts = 1) equals gs_verify_batch. */
int gs_verify_partial(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                      const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                      const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, int rank, int world,
                      gs_gt* out_partial);
int gs_verify_partial_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                          const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                          const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, int rank, int world,
                          gs_gt* out_partial_dev);
/* partials[nparts][count][4] (the all-gathered out_partial arrays, rank-major): entry-wise product over the
 * parts, ONE final exponentiation per ComT entry, comparison with iota_T(target) (PPE: target[count] GT
 * values; the other types carry their target inside a slot, `target` is ignored).  out_ok[count]. */
int gs_verify_finish(gs_ctx* ctx, int type, size_t count, int nparts, const gs_gt* partials, const void* target,
                     uint8_t* out_ok);
int gs_verify_finish_dev(gs_ctx* ctx, int type, size_t count, int nparts, const gs_gt* partials_dev,
                         const void* target_dev, uint8_t* out_ok_dev);

/* The same statement(s) with the statement MSM split by BASE as well: rank r sums only the bases i = r (mod world) into
 * every output and the partial sums (n_out x 2 affine G1 points per statement) are exchanged before the split by slot
 * takes over; the 4 x 576 B Miller partial products are exchanged a second time and every rank finishes.  ONE call runs
 * the whole sharded verification; the two all-gathers go through the caller's transport (NCCL over NVLink via
 * torch.distributed, raw NCCL, MPI ...):
 *     allgather(user, send_dev, recv_dev, bytes) -> 0 once recv_dev[r * bytes ..] holds rank r's send_dev for every r
 * with DEVICE pointers; the context's stream is idle during the callback.  gamma_rows holds ONLY this rank's rows of
 * Gamma: [count][gm][n] with gm = #{i < m : i = rank (mod world)}, row i of Gamma at index i / world -- so a rank uploads
 * 1 / world of the statement.  With world = 1 (allgather = a device copy) this equals gs_verify_batch.  Replaces the
 * Rayon parallelism of left_mul (src/data_structures.rs:708-728) inside verify (src/verifier.rs:39-42). */
typedef int (*gs_allgather_fn)(void* user, const void* send_dev, void* recv_dev, size_t bytes_per_rank);
int gs_verify_sharded(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts, const void* b_consts,
                      const gs_fr* gamma_rows, const void* target, const gs_com1* xcoms, const gs_com2* ycoms,
                      const gs_com2* pi, const gs_com1* theta, int rank, int world, gs_allgather_fn allgather, void* user,
                      uint8_t* out_ok);

/* Randomised batch verification -- SURVEY.md §8f.4, an OPT-IN that the reference does not have (its `verify` is
 * src/verifier.rs:23-157, one proof at a time, four final exponentiations each).  ONE verdict for the whole batch:
 * *out_all_ok = 1 iff every proof verifies, except with probability <= 2^-62 over `rho`.  Not bit-comparable with the
 * reference's per-proof booleans: when the answer is 0 the caller learns which proofs failed from gs_verify_batch.
 * rho[2*count + 1]: 64-bit words from the CALLER's cryptographic RNG, unknown to whoever made the proofs
 * (the low 63 bits of rho[2p], rho[2p+1] weight the two Com1 coordinates of proof p, rho[2*count] the Com2 coordinates of
 * all of them).
 * The four ComT entries of all proofs are folded into a single pairing product: one Miller pair per slot and one final
 * exponentiation per call (csrc/verify.cu, "randomised batch verification").  Soundness needs what the exact
 * verifier assumes too: every point in its prime-order group (gs_g1/g2_decompress check it) and, for PPE, every target
 * in GT (gs_gt_from_bytes checks it).  Arrays as for gs_verify_batch; the _dev variant takes device arrays (rho and
 * nothing else on the host) and writes one byte of device memory. */
int gs_verify_batch_rand(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                         const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                         const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const uint64_t* rho,
                         uint8_t* out_all_ok);
int gs_verify_batch_rand_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                             const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                             const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const uint64_t* rho,
                             uint8_t* out_all_ok_dev);

/* Randomised PER-PROOF verification, an opt-in like gs_verify_batch_rand: out_ok[p] = 1 iff proof p verifies, except
 * with probability <= 2^-62 over `rho` for every bad proof on its own.  The four ComT entries of proof p are folded with
 * the same weights as gs_verify_batch_rand (sigma_p, tau_p = low 63 bits of rho[2p], rho[2p+1]; beta = rho[2*count],
 * shared by the call), and nothing is multiplied across proofs: proof p is accepted iff
 *     FE( prod_k e( sigma_p X_k.0 + tau_p X_k.1 ,  beta Y_k.0 + Y_k.1 ) ) == t_p^tau_p   (PPE; 1 for the other types)
 * over the slots (X_k, Y_k) of the exact verifier -- one Miller pair per slot and ONE final exponentiation per proof
 * (csrc/verify.cu, "randomised per-proof verification").  A proof that fails the exact check passes only if a non-zero
 * polynomial of degree 2 in (sigma_p, tau_p, beta) vanishes.  Preconditions, arrays and return codes as for
 * gs_verify_batch_rand; count == 0 returns GS_OK and writes nothing; a null rho or output of a non-empty call is
 * GS_EARG.  An all-zero rho accepts everything (the check is then vacuous).  The verdicts are not bit-comparable with the
 * reference's.  The _dev variant takes device arrays (rho stays on the host) and writes `count` bytes of device memory,
 * asynchronously on gs_stream(). */
int gs_verify_each_rand(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                        const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                        const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const uint64_t* rho,
                        uint8_t* out_ok);
int gs_verify_each_rand_dev(gs_ctx* ctx, int type, size_t count, size_t m, size_t n, const void* a_consts,
                            const void* b_consts, const gs_fr* gamma, const void* target, const gs_com1* xcoms,
                            const gs_com2* ycoms, const gs_com2* pi, const gs_com1* theta, const uint64_t* rho,
                            uint8_t* out_ok_dev);

/* ---- ComT (src/data_structures.rs) ------------------------------------------------------- */
/* ComT::pairing :484-491, batched: out[i] = F(xs[i], ys[i]) (4 full pairings each) */
int gs_comt_pairing(gs_ctx* ctx, size_t count, const gs_com1* xs, const gs_com2* ys, gs_comt* out);
/* ComT::pairing_sum :494-502: out = sum_i F(xs[i], ys[i]) (one final exponentiation per entry) */
int gs_comt_pairing_sum(gs_ctx* ctx, size_t k, const gs_com1* xs, const gs_com2* ys, gs_comt* out);
/* The four iota_T maps :509-540 (type selects linear_map_PPE / _MSMEG1 / _MSMEG2 / _quad) */
int gs_comt_linear_map(gs_ctx* ctx, int type, const void* target, gs_comt* out);
/* E::pairing batched: out[i] = e(ps[i], qs[i]) */
int gs_pairing(gs_ctx* ctx, size_t count, const gs_g1* ps, const gs_g2* qs, gs_gt* out);

/* ---- commitment-group arithmetic (src/data_structures.rs:162-255, 391-479) ----------------------- */
/* Entry-wise Add / Sub / Neg over n elements and Sum (fold from zero: n = 0 gives the identity) for
 * Com1 = G1 x G1, Com2 = G2 x G2 (impl_base_commit_groups! :162-255) and ComT = GT^4 (:391-479), where GT is
 * written additively as arkworks' PairingOutput does: add = Fp12 product, neg = conjugate. */
int gs_com1_add(gs_ctx* ctx, size_t n, const gs_com1* a, const gs_com1* b, gs_com1* out);
int gs_com1_sub(gs_ctx* ctx, size_t n, const gs_com1* a, const gs_com1* b, gs_com1* out);
int gs_com1_neg(gs_ctx* ctx, size_t n, const gs_com1* a, gs_com1* out);
int gs_com1_sum(gs_ctx* ctx, size_t n, const gs_com1* a, gs_com1* out);
int gs_com2_add(gs_ctx* ctx, size_t n, const gs_com2* a, const gs_com2* b, gs_com2* out);
int gs_com2_sub(gs_ctx* ctx, size_t n, const gs_com2* a, const gs_com2* b, gs_com2* out);
int gs_com2_neg(gs_ctx* ctx, size_t n, const gs_com2* a, gs_com2* out);
int gs_com2_sum(gs_ctx* ctx, size_t n, const gs_com2* a, gs_com2* out);
int gs_comt_add(gs_ctx* ctx, size_t n, const gs_comt* a, const gs_comt* b, gs_comt* out);
int gs_comt_sub(gs_ctx* ctx, size_t n, const gs_comt* a, const gs_comt* b, gs_comt* out);
int gs_comt_neg(gs_ctx* ctx, size_t n, const gs_comt* a, gs_comt* out);
int gs_comt_sum(gs_ctx* ctx, size_t n, const gs_comt* a, gs_comt* out);
/* Matrix<Fr> element-wise parts of the Mat trait (:771-807): add, (sub), neg, scalar_mul over n entries */
int gs_fr_add(gs_ctx* ctx, size_t n, const gs_fr* a, const gs_fr* b, gs_fr* out);
int gs_fr_sub(gs_ctx* ctx, size_t n, const gs_fr* a, const gs_fr* b, gs_fr* out);
int gs_fr_neg(gs_ctx* ctx, size_t n, const gs_fr* a, gs_fr* out);
int gs_fr_scale(gs_ctx* ctx, size_t n, const gs_fr* s, const gs_fr* a, gs_fr* out);

/* ---- wire formats (ark-serialize as derived at generator.rs:35, commit.rs:18-28, prove.rs:55-61) ---- */
/* Point compression in ark-bls12-381's zcash / IETF encoding: G1 48 B = big-endian x, G2 96 B = x.c1 || x.c0,
 * top bits of byte 0: 0x80 compressed, 0x40 infinity, 0x20 y is the lexicographically largest of {y, -y}.
 * Decompression validates like CanonicalDeserialize with Validate::Yes: out_ok[i] = 0 (and out[i] = identity)
 * when the flag byte is not a compressed encoding, x >= p, x is not on the curve, or -- with check_subgroup
 * != 0 -- the point is outside the order-r subgroup.  A set infinity flag yields the identity. */
int gs_g1_compress(gs_ctx* ctx, size_t n, const gs_g1* pts, uint8_t* out /* 48 n */);
int gs_g1_decompress(gs_ctx* ctx, size_t n, const uint8_t* in, int check_subgroup, gs_g1* out, uint8_t* out_ok);
int gs_g2_compress(gs_ctx* ctx, size_t n, const gs_g2* pts, uint8_t* out /* 96 n */);
int gs_g2_decompress(gs_ctx* ctx, size_t n, const uint8_t* in, int check_subgroup, gs_g2* out, uint8_t* out_ok);
/* serialize_uncompressed: G1 96 B = x || y, G2 192 B = x.c1 || x.c0 || y.c1 || y.c0 (big-endian), byte 0: 0x80 clear,
 * 0x40 infinity.  Reading validates coordinates < p, the curve equation and (check_subgroup != 0) the subgroup. */
int gs_g1_serialize_uncompressed(gs_ctx* ctx, size_t n, const gs_g1* pts, uint8_t* out /* 96 n */);
int gs_g1_deserialize_uncompressed(gs_ctx* ctx, size_t n, const uint8_t* in, int check_subgroup, gs_g1* out, uint8_t* out_ok);
int gs_g2_serialize_uncompressed(gs_ctx* ctx, size_t n, const gs_g2* pts, uint8_t* out /* 192 n */);
int gs_g2_deserialize_uncompressed(gs_ctx* ctx, size_t n, const uint8_t* in, int check_subgroup, gs_g2* out, uint8_t* out_ok);
/* Fr <-> 32 B little-endian canonical integer; GT <-> 12 x 48 B little-endian canonical, tower order.
 * from_bytes rejects integers >= the modulus (out_ok[i] = 0, value zeroed). */
int gs_fr_to_bytes(gs_ctx* ctx, size_t n, const gs_fr* in, uint8_t* out);
int gs_fr_from_bytes(gs_ctx* ctx, size_t n, const uint8_t* in, gs_fr* out, uint8_t* out_ok);
int gs_gt_to_bytes(gs_ctx* ctx, size_t n, const gs_gt* in, uint8_t* out);
int gs_gt_from_bytes(gs_ctx* ctx, size_t n, const uint8_t* in, gs_gt* out, uint8_t* out_ok);

/* ---- Mat (src/data_structures.rs:645-742, 768-913) ---------------------------------------- */
/* out (r x c) = lhs (r x k, Fr) * mat (k x c, Com1) -- Matrix<Com1>::left_mul */
int gs_com1_matmul(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* lhs, const gs_com1* mat, gs_com1* out);
int gs_com2_matmul(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* lhs, const gs_com2* mat, gs_com2* out);
/* out (r x c) = a (r x k) * b (k x c) over Fr -- Matrix<Fr>::right_mul */
int gs_fr_matmul(gs_ctx* ctx, size_t r, size_t k, size_t c, const gs_fr* a, const gs_fr* b, gs_fr* out);

#ifdef __cplusplus
}
#endif
#endif /* GS_B200_H */
