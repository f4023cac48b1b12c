//! Proofs (reference: `src/prover/prove.rs:29-489`).  One `gs_prove` call per equation; the proof randomness T is drawn
//! on the host in the reference's order (row-major, `:123-126`, `:226-227`, `:329-332`, `:440`) and stored in `EquProof.rand`.
use super::commit::*;
use crate::data_structures::{Com1, Com2, Matrix};
use crate::ffi::*;
use crate::generator::CRS;
use crate::statement::*;
use ark_ec::pairing::PairingOutput;
use ark_ff::{UniformRand, Zero};
use ark_serialize::{CanonicalDeserialize, CanonicalSerialize};
use ark_std::rand::Rng;

pub trait Provable<E: Gpu, A1, A2, AT> {
    fn commit_and_prove<CR: Rng>(&self, xvars: &[A1], yvars: &[A2], crs: &CRS<E>, rng: &mut CR) -> CProof<E>;
    fn prove<CR: Rng>(&self, xvars: &[A1], yvars: &[A2], xcoms: &Commit1<E>, ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> EquProof<E>;
}

#[derive(Clone, Debug, PartialEq, Eq, CanonicalSerialize, CanonicalDeserialize)]
pub struct EquProof<E: Gpu> { pub pi: Vec<Com2<E>>, pub theta: Vec<Com1<E>>, pub equ_type: EquType, pub(crate) rand: Matrix<E::ScalarField> }

#[derive(Clone, Debug, PartialEq, Eq)]
pub struct CProof<E: Gpu> { pub xcoms: Commit1<E>, pub ycoms: Commit2<E>, pub equ_proofs: Vec<EquProof<E>> }

/// Shared body: the dimension asserts of the reference, T drawn cy x cx row-major, one `gs_prove`.
/// `a`, `b`, `x`, `y` are the flattened constants / witnesses (G1 / G2 points or Fr, as the type says).
#[allow(clippy::too_many_arguments)]
fn prove_any<E: Gpu, CR: Rng>(ty: EquType, cx: usize, cy: usize, gamma: &Matrix<E::ScalarField>, a: &[u8], b: &[u8], x: &[u8], y: &[u8],
                              m: usize, n: usize, xcoms: &Commit1<E>, ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> EquProof<E> {
    assert_eq!(m, xcoms.rand.len());                      // prove.rs:106-114 and its three siblings
    assert_eq!(gamma.len(), xcoms.rand.len());
    assert_eq!(xcoms.rand[0].len(), cx);
    assert_eq!(n, ycoms.rand.len());
    assert_eq!(gamma[0].len(), ycoms.rand.len());
    assert_eq!(ycoms.rand[0].len(), cy);
    let pf_rand: Matrix<E::ScalarField> = (0..cy).map(|_| (0..cx).map(|_| E::ScalarField::rand(rng)).collect()).collect();
    let (g, r, s, t) = (fr_matrix::<E>(gamma), fr_matrix::<E>(&xcoms.rand), fr_matrix::<E>(&ycoms.rand), fr_matrix::<E>(&pf_rand));
    let mut pi = vec![Com2::<E>::zero().abi(); cx];
    let mut theta = vec![Com1::<E>::zero().abi(); cy];
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_prove(c.raw(), ty.abi(), m, n, a.as_ptr(), b.as_ptr(), g.as_ptr(), x.as_ptr(), y.as_ptr(), r.as_ptr(), s.as_ptr(), t.as_ptr(),
                 pi.as_mut_ptr(), theta.as_mut_ptr())
    }));
    EquProof { pi: pi.iter().map(Com2::from_abi).collect(), theta: theta.iter().map(Com1::from_abi).collect(), equ_type: ty, rand: pf_rand }
}

fn bytes_of<T>(v: &[T]) -> &[u8] { unsafe { std::slice::from_raw_parts(v.as_ptr() as *const u8, std::mem::size_of_val(v)) } }

impl<E: Gpu> Provable<E, E::G1Affine, E::G2Affine, PairingOutput<E>> for PPE<E> {
    fn commit_and_prove<CR: Rng>(&self, xvars: &[E::G1Affine], yvars: &[E::G2Affine], crs: &CRS<E>, rng: &mut CR) -> CProof<E> {
        let xcoms = batch_commit_G1(xvars, crs, rng);                    // RNG order: x rows, y rows, then T (`:82-88`)
        let ycoms = batch_commit_G2(yvars, crs, rng);
        let p = self.prove(xvars, yvars, &xcoms, &ycoms, crs, rng);
        CProof { xcoms, ycoms, equ_proofs: vec![p] }
    }
    fn prove<CR: Rng>(&self, xvars: &[E::G1Affine], yvars: &[E::G2Affine], xcoms: &Commit1<E>, ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> EquProof<E> {
        let (a, b, x, y) = (g1s::<E>(&self.a_consts), g2s::<E>(&self.b_consts), g1s::<E>(xvars), g2s::<E>(yvars));
        prove_any(EquType::PairingProduct, 2, 2, &self.gamma, bytes_of(&a), bytes_of(&b), bytes_of(&x), bytes_of(&y), xvars.len(), yvars.len(), xcoms, ycoms, crs, rng)
    }
}
impl<E: Gpu> Provable<E, E::G1Affine, E::ScalarField, E::G1Affine> for MSMEG1<E> {
    fn commit_and_prove<CR: Rng>(&self, xvars: &[E::G1Affine], scalar_yvars: &[E::ScalarField], crs: &CRS<E>, rng: &mut CR) -> CProof<E> {
        let xcoms = batch_commit_G1(xvars, crs, rng);
        let ycoms = batch_commit_scalar_to_B2(scalar_yvars, crs, rng);
        let p = self.prove(xvars, scalar_yvars, &xcoms, &ycoms, crs, rng);
        CProof { xcoms, ycoms, equ_proofs: vec![p] }
    }
    fn prove<CR: Rng>(&self, xvars: &[E::G1Affine], scalar_yvars: &[E::ScalarField], xcoms: &Commit1<E>, ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> EquProof<E> {
        let (a, b, x, y) = (g1s::<E>(&self.a_consts), frs::<E>(&self.b_consts), g1s::<E>(xvars), frs::<E>(scalar_yvars));
        prove_any(EquType::MultiScalarG1, 2, 1, &self.gamma, bytes_of(&a), bytes_of(&b), bytes_of(&x), bytes_of(&y), xvars.len(), scalar_yvars.len(), xcoms, ycoms, crs, rng)
    }
}
impl<E: Gpu> Provable<E, E::ScalarField, E::G2Affine, E::G2Affine> for MSMEG2<E> {
    fn commit_and_prove<CR: Rng>(&self, scalar_xvars: &[E::ScalarField], yvars: &[E::G2Affine], crs: &CRS<E>, rng: &mut CR) -> CProof<E> {
        let xcoms = batch_commit_scalar_to_B1(scalar_xvars, crs, rng);
        let ycoms = batch_commit_G2(yvars, crs, rng);
        let p = self.prove(scalar_xvars, yvars, &xcoms, &ycoms, crs, rng);
        CProof { xcoms, ycoms, equ_proofs: vec![p] }
    }
    fn prove<CR: Rng>(&self, scalar_xvars: &[E::ScalarField], yvars: &[E::G2Affine], xcoms: &Commit1<E>, ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> EquProof<E> {
        let (a, b, x, y) = (frs::<E>(&self.a_consts), g2s::<E>(&self.b_consts), frs::<E>(scalar_xvars), g2s::<E>(yvars));
        prove_any(EquType::MultiScalarG2, 1, 2, &self.gamma, bytes_of(&a), bytes_of(&b), bytes_of(&x), bytes_of(&y), scalar_xvars.len(), yvars.len(), xcoms, ycoms, crs, rng)
    }
}
impl<E: Gpu> Provable<E, E::ScalarField, E::ScalarField, E::ScalarField> for QuadEqu<E> {
    fn commit_and_prove<CR: Rng>(&self, scalar_xvars: &[E::ScalarField], scalar_yvars: &[E::ScalarField], crs: &CRS<E>, rng: &mut CR) -> CProof<E> {
        let xcoms = batch_commit_scalar_to_B1(scalar_xvars, crs, rng);
        let ycoms = batch_commit_scalar_to_B2(scalar_yvars, crs, rng);
        let p = self.prove(scalar_xvars, scalar_yvars, &xcoms, &ycoms, crs, rng);
        CProof { xcoms, ycoms, equ_proofs: vec![p] }
    }
    fn prove<CR: Rng>(&self, scalar_xvars: &[E::ScalarField], scalar_yvars: &[E::ScalarField], xcoms: &Commit1<E>, ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> EquProof<E> {
        let (a, b, x, y) = (frs::<E>(&self.a_consts), frs::<E>(&self.b_consts), frs::<E>(scalar_xvars), frs::<E>(scalar_yvars));
        prove_any(EquType::Quadratic, 1, 1, &self.gamma, bytes_of(&a), bytes_of(&b), bytes_of(&x), bytes_of(&y), scalar_xvars.len(), scalar_yvars.len(), xcoms, ycoms, crs, rng)
    }
}

/// Not in the reference: all equations of ONE type over shared witnesses (a multi-equation statement) in one GPU pass
/// (`gs_prove_batch`, shared_vars = 1).  Results equal `equations.iter().map(|e| e.prove(..))` with the same RNG stream.
pub fn prove_statement_ppe<E: Gpu, CR: Rng>(equations: &[PPE<E>], xvars: &[E::G1Affine], yvars: &[E::G2Affine], xcoms: &Commit1<E>,
                                            ycoms: &Commit2<E>, crs: &CRS<E>, rng: &mut CR) -> Vec<EquProof<E>> {
    let (m, n, count) = (xvars.len(), yvars.len(), equations.len());
    let mut a = Vec::new(); let mut b = Vec::new(); let mut g = Vec::new(); let mut t = Vec::new(); let mut rands = Vec::new();
    for e in equations {
        assert_eq!((e.a_consts.len(), e.b_consts.len(), e.gamma.len()), (n, m, m));
        a.extend(g1s::<E>(&e.a_consts)); b.extend(g2s::<E>(&e.b_consts)); g.extend(fr_matrix::<E>(&e.gamma));
        let pf: Matrix<E::ScalarField> = (0..2).map(|_| (0..2).map(|_| E::ScalarField::rand(rng)).collect()).collect();
        t.extend(fr_matrix::<E>(&pf)); rands.push(pf);
    }
    let (x, y, r, s) = (g1s::<E>(xvars), g2s::<E>(yvars), fr_matrix::<E>(&xcoms.rand), fr_matrix::<E>(&ycoms.rand));
    let mut pi = vec![Com2::<E>::zero().abi(); 2 * count];
    let mut theta = vec![Com1::<E>::zero().abi(); 2 * count];
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_prove_batch(c.raw(), 0, count, m, n, bytes_of(&a).as_ptr(), bytes_of(&b).as_ptr(), g.as_ptr(), bytes_of(&x).as_ptr(),
                       bytes_of(&y).as_ptr(), r.as_ptr(), s.as_ptr(), t.as_ptr(), 1, pi.as_mut_ptr(), theta.as_mut_ptr())
    }));
    rands.into_iter().enumerate().map(|(i, rand)| EquProof {
        pi: pi[2 * i..2 * i + 2].iter().map(Com2::from_abi).collect(), theta: theta[2 * i..2 * i + 2].iter().map(Com1::from_abi).collect(),
        equ_type: EquType::PairingProduct, rand }).collect()
}

/// Not in the reference: a fresh-looking CProof of the same PPE statement from `proof` alone, without the witnesses or the
/// old randomness (`gs_rerandomize`; Belenkiy et al., CRYPTO 2009).  RNG order: R' (m x 2) rows, S' (n x 2) rows, then T'
/// (2 x 2), row-major -- commit_and_prove's.  The openings are unknown to the caller, so the returned `rand` matrices are empty.
pub fn rerandomize_ppe<E: Gpu, CR: Rng>(equ: &PPE<E>, proof: &CProof<E>, crs: &CRS<E>, rng: &mut CR) -> CProof<E> {
    let (m, n) = (proof.xcoms.coms.len(), proof.ycoms.coms.len());
    assert_eq!(proof.equ_proofs.len(), 1);
    assert_eq!((equ.a_consts.len(), equ.b_consts.len(), equ.gamma.len()), (n, m, m));
    let mut draw = |rows: usize| -> Matrix<E::ScalarField> { (0..rows).map(|_| (0..2).map(|_| E::ScalarField::rand(rng)).collect()).collect() };
    let (r2, s2, t2) = (draw(m), draw(n), draw(2));
    let ep = &proof.equ_proofs[0];
    let (a, b, g) = (g1s::<E>(&equ.a_consts), g2s::<E>(&equ.b_consts), fr_matrix::<E>(&equ.gamma));
    let xc: Vec<GsCom1> = proof.xcoms.coms.iter().map(|c| c.abi()).collect();
    let yc: Vec<GsCom2> = proof.ycoms.coms.iter().map(|c| c.abi()).collect();
    let pi: Vec<GsCom2> = ep.pi.iter().map(|c| c.abi()).collect();
    let th: Vec<GsCom1> = ep.theta.iter().map(|c| c.abi()).collect();
    let (r, s, t) = (fr_matrix::<E>(&r2), fr_matrix::<E>(&s2), fr_matrix::<E>(&t2));
    let mut oxc = vec![Com1::<E>::zero().abi(); m];
    let mut oyc = vec![Com2::<E>::zero().abi(); n];
    let mut opi = vec![Com2::<E>::zero().abi(); 2];
    let mut oth = vec![Com1::<E>::zero().abi(); 2];
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_rerandomize(c.raw(), 0, m, n, bytes_of(&a).as_ptr(), bytes_of(&b).as_ptr(), g.as_ptr(), xc.as_ptr(), yc.as_ptr(),
                       pi.as_ptr(), th.as_ptr(), r.as_ptr(), s.as_ptr(), t.as_ptr(), oxc.as_mut_ptr(), oyc.as_mut_ptr(),
                       opi.as_mut_ptr(), oth.as_mut_ptr())
    }));
    CProof {
        xcoms: Commit1 { coms: oxc.iter().map(Com1::from_abi).collect(), rand: vec![] },
        ycoms: Commit2 { coms: oyc.iter().map(Com2::from_abi).collect(), rand: vec![] },
        equ_proofs: vec![EquProof { pi: opi.iter().map(Com2::from_abi).collect(), theta: oth.iter().map(Com1::from_abi).collect(),
                                    equ_type: EquType::PairingProduct, rand: vec![] }],
    }
}
