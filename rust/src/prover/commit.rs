//! Commitments (reference: `src/prover/commit.rs:12-256`).  Randomness is drawn on the host, one row per variable in
//! order (`:85-88`, `:132-138`), kept in `Commit*.rand` (it is part of the serialisation) and passed to the GPU.
use crate::data_structures::{Com1, Com2, Matrix};
use crate::ffi::*;
use crate::generator::CRS;
use ark_ff::{UniformRand, Zero};
use ark_serialize::{CanonicalDeserialize, CanonicalSerialize};
use ark_std::rand::Rng;
use std::fmt::Debug;

pub trait Commit: Eq + Debug { fn append(&mut self, other: &mut Self); }

#[derive(Clone, Debug, CanonicalSerialize, CanonicalDeserialize)]
pub struct Commit1<E: Gpu> { pub coms: Vec<Com1<E>>, pub(crate) rand: Matrix<E::ScalarField> }
#[derive(Clone, Debug, CanonicalSerialize, CanonicalDeserialize)]
pub struct Commit2<E: Gpu> { pub coms: Vec<Com2<E>>, pub(crate) rand: Matrix<E::ScalarField> }

macro_rules! commit_impl {
    ($t:ident) => {
        impl<E: Gpu> PartialEq for $t<E> { fn eq(&self, o: &Self) -> bool { self.coms == o.coms && self.rand == o.rand } }
        impl<E: Gpu> Eq for $t<E> {}
        impl<E: Gpu> Commit for $t<E> {
            fn append(&mut self, other: &mut Self) {                       // `:42-51`: one randomness row per commitment
                assert_eq!(self.coms.len(), self.rand.len());
                assert_eq!(other.coms.len(), other.rand.len());
                self.coms.append(&mut other.coms);
                self.rand.append(&mut other.rand);
            }
        }
    };
}
commit_impl!(Commit1);
commit_impl!(Commit2);

fn draw_rows<E: Gpu, CR: Rng>(rows: usize, cols: usize, rng: &mut CR) -> Matrix<E::ScalarField> {
    (0..rows).map(|_| (0..cols).map(|_| E::ScalarField::rand(rng)).collect()).collect()
}

/// c_i = iota_1(X_i) + R[i][0] u1 + R[i][1] u2, R is m x 2 (`:78-100`)
pub fn batch_commit_G1<CR: Rng, E: Gpu>(xvars: &[E::G1Affine], key: &CRS<E>, rng: &mut CR) -> Commit1<E> {
    let rand = draw_rows::<E, CR>(xvars.len(), 2, rng);
    let (x, r) = (g1s::<E>(xvars), fr_matrix::<E>(&rand));
    let mut out = vec![Com1::<E>::zero().abi(); xvars.len()];
    with_crs(&key.abi(), |c| check(c, unsafe { gs_batch_commit_g1(c.raw(), x.len(), x.as_ptr(), r.as_ptr(), out.as_mut_ptr()) }));
    Commit1 { coms: out.iter().map(Com1::from_abi).collect(), rand }
}
/// (`:178-200`)
pub fn batch_commit_G2<CR: Rng, E: Gpu>(yvars: &[E::G2Affine], key: &CRS<E>, rng: &mut CR) -> Commit2<E> {
    let rand = draw_rows::<E, CR>(yvars.len(), 2, rng);
    let (y, r) = (g2s::<E>(yvars), fr_matrix::<E>(&rand));
    let mut out = vec![Com2::<E>::zero().abi(); yvars.len()];
    with_crs(&key.abi(), |c| check(c, unsafe { gs_batch_commit_g2(c.raw(), y.len(), y.as_ptr(), r.as_ptr(), out.as_mut_ptr()) }));
    Commit2 { coms: out.iter().map(Com2::from_abi).collect(), rand }
}
/// c_i = x_i W1 + r_i u1, r is m' x 1 (`:125-156`)
pub fn batch_commit_scalar_to_B1<CR: Rng, E: Gpu>(scalar_xvars: &[E::ScalarField], key: &CRS<E>, rng: &mut CR) -> Commit1<E> {
    let rand = draw_rows::<E, CR>(scalar_xvars.len(), 1, rng);
    let (x, r) = (frs::<E>(scalar_xvars), fr_matrix::<E>(&rand));
    let mut out = vec![Com1::<E>::zero().abi(); x.len()];
    with_crs(&key.abi(), |c| check(c, unsafe { gs_batch_commit_scalar_b1(c.raw(), x.len(), x.as_ptr(), r.as_ptr(), out.as_mut_ptr()) }));
    Commit1 { coms: out.iter().map(Com1::from_abi).collect(), rand }
}
/// (`:225-256`)
pub fn batch_commit_scalar_to_B2<CR: Rng, E: Gpu>(scalar_yvars: &[E::ScalarField], key: &CRS<E>, rng: &mut CR) -> Commit2<E> {
    let rand = draw_rows::<E, CR>(scalar_yvars.len(), 1, rng);
    let (y, r) = (frs::<E>(scalar_yvars), fr_matrix::<E>(&rand));
    let mut out = vec![Com2::<E>::zero().abi(); y.len()];
    with_crs(&key.abi(), |c| check(c, unsafe { gs_batch_commit_scalar_b2(c.raw(), y.len(), y.as_ptr(), r.as_ptr(), out.as_mut_ptr()) }));
    Commit2 { coms: out.iter().map(Com2::from_abi).collect(), rand }
}
// single-element forms (`:59-75`, `:103-122`, `:159-175`, `:203-222`): a batch of one draws the same values in the same order
pub fn commit_G1<CR: Rng, E: Gpu>(xvar: &E::G1Affine, key: &CRS<E>, rng: &mut CR) -> Commit1<E> { batch_commit_G1(&[*xvar], key, rng) }
pub fn commit_G2<CR: Rng, E: Gpu>(yvar: &E::G2Affine, key: &CRS<E>, rng: &mut CR) -> Commit2<E> { batch_commit_G2(&[*yvar], key, rng) }
pub fn commit_scalar_to_B1<CR: Rng, E: Gpu>(x: &E::ScalarField, key: &CRS<E>, rng: &mut CR) -> Commit1<E> { batch_commit_scalar_to_B1(&[*x], key, rng) }
pub fn commit_scalar_to_B2<CR: Rng, E: Gpu>(y: &E::ScalarField, key: &CRS<E>, rng: &mut CR) -> Commit2<E> { batch_commit_scalar_to_B2(&[*y], key, rng) }
