//! The FFI boundary: `extern "C"` declarations for every symbol of `include/gs_b200.h`, the `#[repr(C)]`
//! mirror of its plain-data types, a per-thread context, and the conversions between arkworks values and the
//! ABI layout.  arkworks' `Fp<MontBackend<_, N>, N>` holds `BigInt<N>([u64; N])` in Montgomery form -- the
//! ABI's layout exactly -- so field elements are copied limb for limb, never converted.
use ark_bls12_381::{Bls12_381, Fq, Fq12, Fq2, Fq6, Fr, G1Affine, G2Affine};
use ark_ec::{pairing::Pairing, pairing::PairingOutput, AffineRepr};
use ark_ff::{BigInt, PrimeField, Zero};
use std::{cell::RefCell, ffi::CStr, os::raw::c_char};

pub const GS_OK: i32 = 0;
pub const GS_EDIM: i32 = 1;

#[repr(C)] #[derive(Clone, Copy, Default)] pub struct GsFr(pub [u64; 4]);
#[repr(C)] #[derive(Clone, Copy)] pub struct GsG1 { pub x: [u64; 6], pub y: [u64; 6] }
#[repr(C)] #[derive(Clone, Copy)] pub struct GsG2 { pub x: [u64; 12], pub y: [u64; 12] }
#[repr(C)] #[derive(Clone, Copy)] pub struct GsCom1(pub [GsG1; 2]);
#[repr(C)] #[derive(Clone, Copy)] pub struct GsCom2(pub [GsG2; 2]);
#[repr(C)] #[derive(Clone, Copy)] pub struct GsGt(pub [u64; 72]);
#[repr(C)] #[derive(Clone, Copy)] pub struct GsComT(pub [GsGt; 4]);
#[repr(C)] #[derive(Clone, Copy)]
pub struct GsCrs { pub u: [GsCom1; 2], pub v: [GsCom2; 2], pub g1_gen: GsG1, pub g2_gen: GsG2, pub gt_gen: GsGt }
pub enum GsCtx {}
/// `int (*)(void* user, const void* send_dev, void* recv_dev, size_t bytes_per_rank)`: gather `bytes_per_rank` from every rank
/// into `recv_dev` (rank-major); device pointers; return 0 when complete.
pub type GsAllgatherFn = unsafe extern "C" fn(user: *mut std::ffi::c_void, send_dev: *const std::ffi::c_void,
                                              recv_dev: *mut std::ffi::c_void, bytes_per_rank: usize) -> i32;

impl GsG1 { pub const ZERO: GsG1 = GsG1 { x: [0; 6], y: [0; 6] }; }
impl GsG2 { pub const ZERO: GsG2 = GsG2 { x: [0; 12], y: [0; 12] }; }
impl GsGt { pub const ZERO: GsGt = GsGt([0; 72]); }

extern "C" {
    pub fn gs_ctx_create(device: i32, out: *mut *mut GsCtx) -> i32;
    pub fn gs_ctx_destroy(ctx: *mut GsCtx);
    pub fn gs_last_error(ctx: *const GsCtx) -> *const c_char;
    pub fn gs_launch_count(ctx: *const GsCtx) -> u64;
    // generator.rs:81-118
    pub fn gs_crs_generate(ctx: *mut GsCtx, p1: *const GsG1, p2: *const GsG2, a1: *const GsFr, a2: *const GsFr,
                           t1: *const GsFr, t2: *const GsFr, out: *mut GsCrs) -> i32;
    pub fn gs_crs_load(ctx: *mut GsCtx, crs: *const GsCrs) -> i32;
    // prover/commit.rs:78-100, 178-200, 125-156, 225-256
    pub fn gs_batch_commit_g1(ctx: *mut GsCtx, n: usize, x: *const GsG1, rand: *const GsFr, out: *mut GsCom1) -> i32;
    pub fn gs_batch_commit_g2(ctx: *mut GsCtx, n: usize, y: *const GsG2, rand: *const GsFr, out: *mut GsCom2) -> i32;
    pub fn gs_batch_commit_scalar_b1(ctx: *mut GsCtx, n: usize, x: *const GsFr, rand: *const GsFr, out: *mut GsCom1) -> i32;
    pub fn gs_batch_commit_scalar_b2(ctx: *mut GsCtx, n: usize, y: *const GsFr, rand: *const GsFr, out: *mut GsCom2) -> i32;
    // prover/prove.rs:92-488
    pub fn gs_prove(ctx: *mut GsCtx, ty: i32, m: usize, n: usize, a: *const u8, b: *const u8, gamma: *const GsFr,
                    x: *const u8, y: *const u8, x_rand: *const GsFr, y_rand: *const GsFr, pf_rand: *const GsFr,
                    out_pi: *mut GsCom2, out_theta: *mut GsCom1) -> i32;
    pub fn gs_prove_batch(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                          gamma: *const GsFr, x: *const u8, y: *const u8, x_rand: *const GsFr, y_rand: *const GsFr,
                          pf_rand: *const GsFr, shared: i32, out_pi: *mut GsCom2, out_theta: *mut GsCom1) -> i32;
    // not in the reference: a committed proof rerandomised without the witnesses (shared_coms != 0: one set of commitments)
    pub fn gs_rerandomize(ctx: *mut GsCtx, ty: i32, m: usize, n: usize, a: *const u8, b: *const u8, gamma: *const GsFr,
                          xcoms: *const GsCom1, ycoms: *const GsCom2, pi: *const GsCom2, theta: *const GsCom1,
                          x_rand: *const GsFr, y_rand: *const GsFr, pf_rand: *const GsFr, out_xcoms: *mut GsCom1,
                          out_ycoms: *mut GsCom2, out_pi: *mut GsCom2, out_theta: *mut GsCom1) -> i32;
    pub fn gs_rerandomize_batch(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                                gamma: *const GsFr, xcoms: *const GsCom1, ycoms: *const GsCom2, pi: *const GsCom2,
                                theta: *const GsCom1, x_rand: *const GsFr, y_rand: *const GsFr, pf_rand: *const GsFr,
                                shared_coms: i32, out_xcoms: *mut GsCom1, out_ycoms: *mut GsCom2, out_pi: *mut GsCom2,
                                out_theta: *mut GsCom1) -> i32;
    // not in the reference: commitments opened with the binding key's trapdoor (xkey = a1, ykey = a2 of gs_crs_generate)
    pub fn gs_extract(ctx: *mut GsCtx, nx: usize, xcoms: *const GsCom1, xkey: *const GsFr, ny: usize, ycoms: *const GsCom2,
                      ykey: *const GsFr, out_x: *mut GsG1, out_y: *mut GsG2) -> i32;
    // verifier.rs:23-157
    pub fn gs_verify_batch(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                           gamma: *const GsFr, target: *const u8, xcoms: *const GsCom1, ycoms: *const GsCom2,
                           pi: *const GsCom2, theta: *const GsCom1, out_ok: *mut u8) -> i32;
    // opt-in, not in the reference: ONE randomised verdict for the whole batch (rho: 2*count + 1 words from the caller's CSPRNG)
    pub fn gs_verify_batch_rand(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                                gamma: *const GsFr, target: *const u8, xcoms: *const GsCom1, ycoms: *const GsCom2,
                                pi: *const GsCom2, theta: *const GsCom1, rho: *const u64, out_all_ok: *mut u8) -> i32;
    // opt-in, not in the reference: ONE randomised verdict PER PROOF (same rho layout; one final exponentiation each)
    pub fn gs_verify_each_rand(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                               gamma: *const GsFr, target: *const u8, xcoms: *const GsCom1, ycoms: *const GsCom2,
                               pi: *const GsCom2, theta: *const GsCom1, rho: *const u64, out_ok: *mut u8) -> i32;
    pub fn gs_verify_partial(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                             gamma: *const GsFr, target: *const u8, xcoms: *const GsCom1, ycoms: *const GsCom2,
                             pi: *const GsCom2, theta: *const GsCom1, rank: i32, world: i32, out_partial: *mut GsGt) -> i32;
    pub fn gs_verify_finish(ctx: *mut GsCtx, ty: i32, count: usize, nparts: i32, partials: *const GsGt,
                            target: *const u8, out_ok: *mut u8) -> i32;
    // the whole sharded verification in one call: statement MSM split by base, Miller pairs by slot; the two all-gathers
    // go through the caller's transport (device pointers), e.g. ncclAllGather on a communicator the host owns
    pub fn gs_verify_sharded(ctx: *mut GsCtx, ty: i32, count: usize, m: usize, n: usize, a: *const u8, b: *const u8,
                             gamma_rows: *const GsFr, target: *const u8, xcoms: *const GsCom1, ycoms: *const GsCom2,
                             pi: *const GsCom2, theta: *const GsCom1, rank: i32, world: i32, allgather: GsAllgatherFn,
                             user: *mut std::ffi::c_void, out_ok: *mut u8) -> i32;
    // data_structures.rs:484-540
    pub fn gs_comt_pairing(ctx: *mut GsCtx, count: usize, xs: *const GsCom1, ys: *const GsCom2, out: *mut GsComT) -> i32;
    pub fn gs_comt_pairing_sum(ctx: *mut GsCtx, k: usize, xs: *const GsCom1, ys: *const GsCom2, out: *mut GsComT) -> i32;
    pub fn gs_comt_linear_map(ctx: *mut GsCtx, ty: i32, target: *const u8, out: *mut GsComT) -> i32;
    pub fn gs_pairing(ctx: *mut GsCtx, count: usize, ps: *const GsG1, qs: *const GsG2, out: *mut GsGt) -> i32;
    // data_structures.rs:645-742, 768-913
    pub fn gs_com1_matmul(ctx: *mut GsCtx, r: usize, k: usize, c: usize, lhs: *const GsFr, mat: *const GsCom1, out: *mut GsCom1) -> i32;
    pub fn gs_com2_matmul(ctx: *mut GsCtx, r: usize, k: usize, c: usize, lhs: *const GsFr, mat: *const GsCom2, out: *mut GsCom2) -> i32;
    pub fn gs_fr_matmul(ctx: *mut GsCtx, r: usize, k: usize, c: usize, a: *const GsFr, b: *const GsFr, out: *mut GsFr) -> i32;
    // data_structures.rs:162-255, 391-479
    pub fn gs_com1_add(ctx: *mut GsCtx, n: usize, a: *const GsCom1, b: *const GsCom1, out: *mut GsCom1) -> i32;
    pub fn gs_com1_sub(ctx: *mut GsCtx, n: usize, a: *const GsCom1, b: *const GsCom1, out: *mut GsCom1) -> i32;
    pub fn gs_com1_neg(ctx: *mut GsCtx, n: usize, a: *const GsCom1, out: *mut GsCom1) -> i32;
    pub fn gs_com1_sum(ctx: *mut GsCtx, n: usize, a: *const GsCom1, out: *mut GsCom1) -> i32;
    pub fn gs_com2_add(ctx: *mut GsCtx, n: usize, a: *const GsCom2, b: *const GsCom2, out: *mut GsCom2) -> i32;
    pub fn gs_com2_sub(ctx: *mut GsCtx, n: usize, a: *const GsCom2, b: *const GsCom2, out: *mut GsCom2) -> i32;
    pub fn gs_com2_neg(ctx: *mut GsCtx, n: usize, a: *const GsCom2, out: *mut GsCom2) -> i32;
    pub fn gs_com2_sum(ctx: *mut GsCtx, n: usize, a: *const GsCom2, out: *mut GsCom2) -> i32;
    pub fn gs_comt_add(ctx: *mut GsCtx, n: usize, a: *const GsComT, b: *const GsComT, out: *mut GsComT) -> i32;
    pub fn gs_comt_sub(ctx: *mut GsCtx, n: usize, a: *const GsComT, b: *const GsComT, out: *mut GsComT) -> i32;
    pub fn gs_comt_neg(ctx: *mut GsCtx, n: usize, a: *const GsComT, out: *mut GsComT) -> i32;
    pub fn gs_comt_sum(ctx: *mut GsCtx, n: usize, a: *const GsComT, out: *mut GsComT) -> i32;
    pub fn gs_fr_add(ctx: *mut GsCtx, n: usize, a: *const GsFr, b: *const GsFr, out: *mut GsFr) -> i32;
    pub fn gs_fr_sub(ctx: *mut GsCtx, n: usize, a: *const GsFr, b: *const GsFr, out: *mut GsFr) -> i32;
    pub fn gs_fr_neg(ctx: *mut GsCtx, n: usize, a: *const GsFr, out: *mut GsFr) -> i32;
    pub fn gs_fr_scale(ctx: *mut GsCtx, n: usize, s: *const GsFr, a: *const GsFr, out: *mut GsFr) -> i32;
    // wire formats (ark-serialize)
    pub fn gs_g1_compress(ctx: *mut GsCtx, n: usize, pts: *const GsG1, out: *mut u8) -> i32;
    pub fn gs_g1_decompress(ctx: *mut GsCtx, n: usize, bytes: *const u8, check_subgroup: i32, out: *mut GsG1, ok: *mut u8) -> i32;
    pub fn gs_g2_compress(ctx: *mut GsCtx, n: usize, pts: *const GsG2, out: *mut u8) -> i32;
    pub fn gs_g2_decompress(ctx: *mut GsCtx, n: usize, bytes: *const u8, check_subgroup: i32, out: *mut GsG2, ok: *mut u8) -> i32;
    pub fn gs_g1_serialize_uncompressed(ctx: *mut GsCtx, n: usize, pts: *const GsG1, out: *mut u8) -> i32;
    pub fn gs_g1_deserialize_uncompressed(ctx: *mut GsCtx, n: usize, bytes: *const u8, check_subgroup: i32, out: *mut GsG1, ok: *mut u8) -> i32;
    pub fn gs_g2_serialize_uncompressed(ctx: *mut GsCtx, n: usize, pts: *const GsG2, out: *mut u8) -> i32;
    pub fn gs_g2_deserialize_uncompressed(ctx: *mut GsCtx, n: usize, bytes: *const u8, check_subgroup: i32, out: *mut GsG2, ok: *mut u8) -> i32;
    pub fn gs_fr_to_bytes(ctx: *mut GsCtx, n: usize, a: *const GsFr, out: *mut u8) -> i32;
    pub fn gs_fr_from_bytes(ctx: *mut GsCtx, n: usize, bytes: *const u8, out: *mut GsFr, ok: *mut u8) -> i32;
    pub fn gs_gt_to_bytes(ctx: *mut GsCtx, n: usize, a: *const GsGt, out: *mut u8) -> i32;
    pub fn gs_gt_from_bytes(ctx: *mut GsCtx, n: usize, bytes: *const u8, out: *mut GsGt, ok: *mut u8) -> i32;
}

// ---------------------------------------------------------------- the curve the engine supports
/// Sealed marker + conversions: implemented for `Bls12_381` only.  Every hot-path function of the crate carries
/// `E: Gpu`, so instantiating the library with another curve does not compile (north star: no CPU fallback).
pub trait Gpu: Pairing {
    fn fr(x: &Self::ScalarField) -> GsFr;
    fn fr_back(x: &GsFr) -> Self::ScalarField;
    fn g1(p: &Self::G1Affine) -> GsG1;
    fn g1_back(p: &GsG1) -> Self::G1Affine;
    fn g2(p: &Self::G2Affine) -> GsG2;
    fn g2_back(p: &GsG2) -> Self::G2Affine;
    fn gt(t: &PairingOutput<Self>) -> GsGt;
    fn gt_back(t: &GsGt) -> PairingOutput<Self>;
}

fn fq_limbs(a: &Fq) -> [u64; 6] { (a.0).0 }                       // Montgomery limbs as stored
fn fq_from(l: &[u64]) -> Fq { Fq::new_unchecked(BigInt::<6>(l.try_into().unwrap())) }
fn fq2_limbs(a: &Fq2) -> [u64; 12] {
    let mut o = [0u64; 12];
    o[..6].copy_from_slice(&fq_limbs(&a.c0));
    o[6..].copy_from_slice(&fq_limbs(&a.c1));
    o
}
fn fq2_from(l: &[u64]) -> Fq2 { Fq2::new(fq_from(&l[..6]), fq_from(&l[6..12])) }

impl Gpu for Bls12_381 {
    fn fr(x: &Fr) -> GsFr { GsFr((x.0).0) }
    fn fr_back(x: &GsFr) -> Fr { Fr::new_unchecked(BigInt::<4>(x.0)) }
    fn g1(p: &G1Affine) -> GsG1 {
        match p.xy() { None => GsG1::ZERO, Some((x, y)) => GsG1 { x: fq_limbs(&x), y: fq_limbs(&y) } }   // identity = all-zero
    }
    fn g1_back(p: &GsG1) -> G1Affine {
        if p.x == [0; 6] && p.y == [0; 6] { G1Affine::zero() } else { G1Affine::new_unchecked(fq_from(&p.x), fq_from(&p.y)) }
    }
    fn g2(p: &G2Affine) -> GsG2 {
        match p.xy() { None => GsG2::ZERO, Some((x, y)) => GsG2 { x: fq2_limbs(&x), y: fq2_limbs(&y) } }
    }
    fn g2_back(p: &GsG2) -> G2Affine {
        if p.x == [0; 12] && p.y == [0; 12] { G2Affine::zero() } else { G2Affine::new_unchecked(fq2_from(&p.x), fq2_from(&p.y)) }
    }
    fn gt(t: &PairingOutput<Bls12_381>) -> GsGt {                    // tower order c0.c0.c0, c0.c0.c1, c0.c1.c0, ...
        let f: &Fq12 = &t.0;
        let mut o = [0u64; 72];
        for (i, c2) in [&f.c0.c0, &f.c0.c1, &f.c0.c2, &f.c1.c0, &f.c1.c1, &f.c1.c2].iter().enumerate() {
            o[12 * i..12 * i + 12].copy_from_slice(&fq2_limbs(c2));
        }
        GsGt(o)
    }
    fn gt_back(t: &GsGt) -> PairingOutput<Bls12_381> {
        let c = |i: usize| fq2_from(&t.0[12 * i..12 * i + 12]);
        PairingOutput(Fq12::new(Fq6::new(c(0), c(1), c(2)), Fq6::new(c(3), c(4), c(5))))
    }
}

// ---------------------------------------------------------------- context: one per thread and GPU (Send, not Sync)
pub struct Ctx { raw: *mut GsCtx, loaded: RefCell<Option<Vec<u64>>> }

impl Ctx {
    pub fn new(device: i32) -> Ctx {
        let mut raw = std::ptr::null_mut();
        let rc = unsafe { gs_ctx_create(device, &mut raw) };
        assert!(rc == GS_OK && !raw.is_null(), "gs_ctx_create({device}) failed: a CUDA device is required (no CPU fallback)");
        Ctx { raw, loaded: RefCell::new(None) }
    }
    pub fn raw(&self) -> *mut GsCtx { self.raw }
    pub fn last_error(&self) -> String { unsafe { CStr::from_ptr(gs_last_error(self.raw)) }.to_string_lossy().into_owned() }
    /// Makes `crs` the context's key unless it already is (compared by its limbs): `gs_crs_load`.
    pub fn use_crs(&self, crs: &GsCrs) {
        let key: Vec<u64> = unsafe { std::slice::from_raw_parts(crs as *const GsCrs as *const u64, std::mem::size_of::<GsCrs>() / 8) }.to_vec();
        if self.loaded.borrow().as_ref() == Some(&key) { return; }
        check(self, unsafe { gs_crs_load(self.raw, crs) });
        *self.loaded.borrow_mut() = Some(key);
    }
}
impl Drop for Ctx { fn drop(&mut self) { unsafe { gs_ctx_destroy(self.raw) } } }

thread_local! { pub static CTX: Ctx = Ctx::new(std::env::var("GS_B200_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0)); }

/// `GS_EDIM` is the reference's `assert_eq!` panic; every other code is a hard failure as well.
pub fn check(c: &Ctx, rc: i32) { if rc != GS_OK { panic!("gs_b200 error {rc}: {}", c.last_error()); } }

/// Runs `f` with the thread's context after making `crs` current.
pub fn with_crs<R>(crs: &GsCrs, f: impl FnOnce(&Ctx) -> R) -> R { CTX.with(|c| { c.use_crs(crs); f(c) }) }
pub fn with_ctx<R>(f: impl FnOnce(&Ctx) -> R) -> R { CTX.with(|c| f(c)) }

pub fn frs<E: Gpu>(v: &[E::ScalarField]) -> Vec<GsFr> { v.iter().map(E::fr).collect() }
pub fn fr_matrix<E: Gpu>(m: &[Vec<E::ScalarField>]) -> Vec<GsFr> { m.iter().flatten().map(E::fr).collect() }
pub fn g1s<E: Gpu>(v: &[E::G1Affine]) -> Vec<GsG1> { v.iter().map(E::g1).collect() }
pub fn g2s<E: Gpu>(v: &[E::G2Affine]) -> Vec<GsG2> { v.iter().map(E::g2).collect() }
pub fn is_zero_fr<E: Gpu>(x: &E::ScalarField) -> bool { x.is_zero() }
pub fn modulus_bits<E: Gpu>() -> u32 { E::ScalarField::MODULUS_BIT_SIZE }
