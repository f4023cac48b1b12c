//! Verification (reference: `src/verifier.rs:18-157`): one `gs_verify_batch` call with count = 1 per `verify`, plus the
//! batched form a service uses.  The GPU evaluates lhs - rhs as ONE pairing product per ComT entry (4 final
//! exponentiations instead of the reference's 20); the boolean is the same.
use crate::data_structures::{com1s, com2s};
use crate::ffi::*;
use crate::generator::CRS;
use crate::prover::CProof;
use crate::statement::*;

pub trait Verifiable<E: Gpu> { fn verify(&self, com_proof: &CProof<E>, crs: &CRS<E>) -> bool; }

fn bytes_of<T>(v: &[T]) -> &[u8] { unsafe { std::slice::from_raw_parts(v.as_ptr() as *const u8, std::mem::size_of_val(v)) } }

#[allow(clippy::too_many_arguments)]
fn verify_any<E: Gpu>(ty: EquType, a: &[u8], b: &[u8], gamma: &[Vec<E::ScalarField>], target: &[u8], proof: &CProof<E>, crs: &CRS<E>) -> bool {
    assert_eq!(proof.equ_proofs.len(), 1);                               // verifier.rs:25-26
    assert_eq!(ty, proof.equ_proofs[0].equ_type);
    let (m, n) = (proof.xcoms.coms.len(), proof.ycoms.coms.len());
    let (g, xc, yc) = (fr_matrix::<E>(gamma), com1s(&proof.xcoms.coms), com2s(&proof.ycoms.coms));
    let (pi, th) = (com2s(&proof.equ_proofs[0].pi), com1s(&proof.equ_proofs[0].theta));
    let mut ok = 0u8;
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_verify_batch(c.raw(), ty.abi(), 1, m, n, a.as_ptr(), b.as_ptr(), g.as_ptr(), target.as_ptr(), xc.as_ptr(), yc.as_ptr(),
                        pi.as_ptr(), th.as_ptr(), &mut ok)
    }));
    ok == 1
}

impl<E: Gpu> Verifiable<E> for PPE<E> {
    fn verify(&self, p: &CProof<E>, crs: &CRS<E>) -> bool {
        let (a, b, t) = (g1s::<E>(&self.a_consts), g2s::<E>(&self.b_consts), [E::gt(&self.target)]);
        verify_any(EquType::PairingProduct, bytes_of(&a), bytes_of(&b), &self.gamma, bytes_of(&t), p, crs)
    }
}
impl<E: Gpu> Verifiable<E> for MSMEG1<E> {
    fn verify(&self, p: &CProof<E>, crs: &CRS<E>) -> bool {
        let (a, b, t) = (g1s::<E>(&self.a_consts), frs::<E>(&self.b_consts), [E::g1(&self.target)]);
        verify_any(EquType::MultiScalarG1, bytes_of(&a), bytes_of(&b), &self.gamma, bytes_of(&t), p, crs)
    }
}
impl<E: Gpu> Verifiable<E> for MSMEG2<E> {
    fn verify(&self, p: &CProof<E>, crs: &CRS<E>) -> bool {
        let (a, b, t) = (frs::<E>(&self.a_consts), g2s::<E>(&self.b_consts), [E::g2(&self.target)]);
        verify_any(EquType::MultiScalarG2, bytes_of(&a), bytes_of(&b), &self.gamma, bytes_of(&t), p, crs)
    }
}
impl<E: Gpu> Verifiable<E> for QuadEqu<E> {
    fn verify(&self, p: &CProof<E>, crs: &CRS<E>) -> bool {
        let (a, b, t) = (frs::<E>(&self.a_consts), frs::<E>(&self.b_consts), [E::fr(&self.target)]);
        verify_any(EquType::Quadratic, bytes_of(&a), bytes_of(&b), &self.gamma, bytes_of(&t), p, crs)
    }
}

/// Not in the reference: `count` independent PPE (equation, proof) pairs of one shape in ONE GPU pass (C5).
/// `randomized = Some(rng)` (a cryptographic RNG the prover cannot predict) turns on the randomised pre-check.
pub fn verify_batch_ppe<E: Gpu>(equations: &[PPE<E>], proofs: &[CProof<E>], crs: &CRS<E>,
                                randomized: Option<&mut dyn ark_std::rand::RngCore>) -> Vec<bool> {
    assert_eq!(equations.len(), proofs.len());
    if equations.is_empty() { return vec![]; }
    let (m, n) = (proofs[0].xcoms.coms.len(), proofs[0].ycoms.coms.len());
    let (mut a, mut b, mut g, mut t) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    let (mut xc, mut yc, mut pi, mut th) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    for (e, p) in equations.iter().zip(proofs) {
        assert_eq!((p.xcoms.coms.len(), p.ycoms.coms.len(), p.equ_proofs.len()), (m, n, 1));
        a.extend(g1s::<E>(&e.a_consts)); b.extend(g2s::<E>(&e.b_consts)); g.extend(fr_matrix::<E>(&e.gamma)); t.push(E::gt(&e.target));
        xc.extend(com1s(&p.xcoms.coms)); yc.extend(com2s(&p.ycoms.coms));
        pi.extend(com2s(&p.equ_proofs[0].pi)); th.extend(com1s(&p.equ_proofs[0].theta));
    }
    // opt-in: one randomised check of the whole batch first (a single folded pairing product, one final exponentiation);
    // only a batch that fails it pays for the exact per-proof pass below, which says WHICH proofs are bad
    if let Some(rng) = randomized {
        let rho: Vec<u64> = (0..2 * equations.len() + 1).map(|_| rng.next_u64()).collect();
        let mut all_ok = 0u8;
        with_crs(&crs.abi(), |c| check(c, unsafe {
            gs_verify_batch_rand(c.raw(), 0, equations.len(), m, n, bytes_of(&a).as_ptr(), bytes_of(&b).as_ptr(), g.as_ptr(),
                                 bytes_of(&t).as_ptr(), xc.as_ptr(), yc.as_ptr(), pi.as_ptr(), th.as_ptr(), rho.as_ptr(), &mut all_ok)
        }));
        if all_ok == 1 { return vec![true; equations.len()]; }
    }
    let mut ok = vec![0u8; equations.len()];
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_verify_batch(c.raw(), 0, ok.len(), m, n, bytes_of(&a).as_ptr(), bytes_of(&b).as_ptr(), g.as_ptr(), bytes_of(&t).as_ptr(),
                        xc.as_ptr(), yc.as_ptr(), pi.as_ptr(), th.as_ptr(), ok.as_mut_ptr())
    }));
    ok.into_iter().map(|x| x == 1).collect()
}

/// Not in the reference: per-proof verdicts of `count` independent PPE (equation, proof) pairs of one shape at close to
/// the randomised cost (gs_verify_each_rand): each proof's four ComT entries are folded with its own weights from `rng`
/// (a cryptographic RNG the prover cannot predict) into one pairing product and ONE final exponentiation.  A bad proof is
/// accepted with probability <= 2^-62, each proof on its own.
pub fn verify_each_ppe_rand<E: Gpu>(equations: &[PPE<E>], proofs: &[CProof<E>], crs: &CRS<E>,
                                    rng: &mut dyn ark_std::rand::RngCore) -> Vec<bool> {
    assert_eq!(equations.len(), proofs.len());
    if equations.is_empty() { return vec![]; }
    let (m, n) = (proofs[0].xcoms.coms.len(), proofs[0].ycoms.coms.len());
    let (mut a, mut b, mut g, mut t) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    let (mut xc, mut yc, mut pi, mut th) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    for (e, p) in equations.iter().zip(proofs) {
        assert_eq!((p.xcoms.coms.len(), p.ycoms.coms.len(), p.equ_proofs.len()), (m, n, 1));
        a.extend(g1s::<E>(&e.a_consts)); b.extend(g2s::<E>(&e.b_consts)); g.extend(fr_matrix::<E>(&e.gamma)); t.push(E::gt(&e.target));
        xc.extend(com1s(&p.xcoms.coms)); yc.extend(com2s(&p.ycoms.coms));
        pi.extend(com2s(&p.equ_proofs[0].pi)); th.extend(com1s(&p.equ_proofs[0].theta));
    }
    let rho: Vec<u64> = (0..2 * equations.len() + 1).map(|_| rng.next_u64()).collect();
    let mut ok = vec![0u8; equations.len()];
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_verify_each_rand(c.raw(), 0, ok.len(), m, n, bytes_of(&a).as_ptr(), bytes_of(&b).as_ptr(), g.as_ptr(),
                            bytes_of(&t).as_ptr(), xc.as_ptr(), yc.as_ptr(), pi.as_ptr(), th.as_ptr(), rho.as_ptr(), ok.as_mut_ptr())
    }));
    ok.into_iter().map(|x| x == 1).collect()
}
