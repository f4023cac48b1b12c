//! Not in the reference: extraction with the binding key (ExtGen / Ext of Groth & Sahai, EUROCRYPT 2008).
//! `generate_crs_with_trapdoor` is `generate_crs` that keeps the trapdoor (a1, a2) instead of dropping it; whoever holds it
//! opens every commitment made under that CRS: X = c.1 - a1 c.0 (`gs_extract`).  Commitments of scalars give x g1 / y g2.
use crate::data_structures::{Com1, Com2};
use crate::ffi::*;
use crate::generator::CRS;
use ark_ff::UniformRand;
use ark_std::rand::Rng;

/// The trapdoor of a binding CRS: u[0] = (p1, a1 p1), v[0] = (p2, a2 p2).
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct ExtractionKey<E: Gpu> { pub a1: E::ScalarField, pub a2: E::ScalarField }

/// `generate_crs` with exactly its draws (p1 <- G1, p2 <- G2, a1, a2, t1, t2 <- Fr), also returning (a1, a2).  The CRS becomes
/// the thread context's current key.
pub fn generate_crs_with_trapdoor<E: Gpu, R: Rng>(rng: &mut R) -> (CRS<E>, ExtractionKey<E>) {
    let p1 = E::G1::rand(rng).into();
    let p2 = E::G2::rand(rng).into();
    let (a1, a2) = (E::ScalarField::rand(rng), E::ScalarField::rand(rng));
    let (t1, t2) = (E::ScalarField::rand(rng), E::ScalarField::rand(rng));
    let (gp1, gp2) = (E::g1(&p1), E::g2(&p2));
    let s = [E::fr(&a1), E::fr(&a2), E::fr(&t1), E::fr(&t2)];
    let mut out = std::mem::MaybeUninit::<GsCrs>::zeroed();
    with_ctx(|c| check(c, unsafe { gs_crs_generate(c.raw(), &gp1, &gp2, &s[0], &s[1], &s[2], &s[3], out.as_mut_ptr()) }));
    (CRS::from_abi(&unsafe { out.assume_init() }), ExtractionKey { a1, a2 })
}

/// The committed G1 values (x g1 for commitments of scalars).  Panics when `key` does not open `crs` (or `crs` is hiding).
pub fn extract_G1<E: Gpu>(coms: &[Com1<E>], key: &ExtractionKey<E>, crs: &CRS<E>) -> Vec<E::G1Affine> {
    let c: Vec<GsCom1> = coms.iter().map(|x| x.abi()).collect();
    let k = E::fr(&key.a1);
    let mut out = vec![GsG1::ZERO; c.len()];
    with_crs(&crs.abi(), |ctx| check(ctx, unsafe {
        gs_extract(ctx.raw(), c.len(), c.as_ptr(), &k, 0, std::ptr::null(), std::ptr::null(), out.as_mut_ptr(), std::ptr::null_mut())
    }));
    out.iter().map(E::g1_back).collect()
}

/// The committed G2 values (y g2 for commitments of scalars).
pub fn extract_G2<E: Gpu>(coms: &[Com2<E>], key: &ExtractionKey<E>, crs: &CRS<E>) -> Vec<E::G2Affine> {
    let c: Vec<GsCom2> = coms.iter().map(|x| x.abi()).collect();
    let k = E::fr(&key.a2);
    let mut out = vec![GsG2::ZERO; c.len()];
    with_crs(&crs.abi(), |ctx| check(ctx, unsafe {
        gs_extract(ctx.raw(), 0, std::ptr::null(), std::ptr::null(), c.len(), c.as_ptr(), &k, std::ptr::null_mut(), out.as_mut_ptr())
    }));
    out.iter().map(E::g2_back).collect()
}
