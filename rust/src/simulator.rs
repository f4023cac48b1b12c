//! Not in the reference: zero-knowledge simulation with the hiding key (Groth & Sahai, EUROCRYPT 2008).
//! `generate_hiding_crs_with_trapdoor` makes the hiding CRS of `generate_crs`'s draws (u[1] - iota_1(g1), v[1] - iota_2(g2))
//! and keeps its trapdoor (t1, t2).  Under it W1 = t1 u[0] and W2 = t2 v[0], so whoever holds the key makes proofs that
//! verify under that CRS without witnesses (`gs_simulate_batch`): for any MSMEG1, MSMEG2 or Quad statement and for PPE
//! statements with target 1.  The simulated proofs are distributed exactly like real ones.
use crate::data_structures::{Com1, Com2};
use crate::ffi::*;
use crate::generator::CRS;
use crate::prover::{CProof, Commit1, Commit2, EquProof};
use crate::statement::{EquType, PPE};
use ark_ec::AffineRepr;
use ark_ff::{UniformRand, Zero};
use ark_std::rand::Rng;

/// The trapdoor of a hiding CRS: W1 = u[1] + iota_1(g1) = t1 u[0], W2 = t2 v[0].
#[derive(Clone, Copy, Debug, PartialEq, Eq)]
pub struct SimulationKey<E: Gpu> { pub t1: E::ScalarField, pub t2: E::ScalarField }

/// The hiding CRS with exactly `generate_crs`'s draws (p1 <- G1, p2 <- G2, a1, a2, t1, t2 <- Fr), also returning (t1, t2).
pub fn generate_hiding_crs_with_trapdoor<E: Gpu, R: Rng>(rng: &mut R) -> (CRS<E>, SimulationKey<E>) {
    let p1 = E::G1::rand(rng).into();
    let p2 = E::G2::rand(rng).into();
    let (a1, a2) = (E::ScalarField::rand(rng), E::ScalarField::rand(rng));
    let (t1, t2) = (E::ScalarField::rand(rng), E::ScalarField::rand(rng));
    let (gp1, gp2) = (E::g1(&p1), E::g2(&p2));
    let s = [E::fr(&a1), E::fr(&a2), E::fr(&t1), E::fr(&t2)];
    let mut out = std::mem::MaybeUninit::<GsCrs>::zeroed();
    with_ctx(|c| check(c, unsafe { gs_crs_generate(c.raw(), &gp1, &gp2, &s[0], &s[1], &s[2], &s[3], out.as_mut_ptr()) }));
    let mut crs = CRS::<E>::from_abi(&unsafe { out.assume_init() });
    crs.u[1] = crs.u[1] - Com1::<E>(<E::G1Affine as AffineRepr>::zero(), crs.g1_gen);
    crs.v[1] = crs.v[1] - Com2::<E>(<E::G2Affine as AffineRepr>::zero(), crs.g2_gen);
    (crs, SimulationKey { t1, t2 })
}

fn bytes_of<T>(v: &[T]) -> &[u8] { unsafe { std::slice::from_raw_parts(v.as_ptr() as *const u8, std::mem::size_of_val(v)) } }

/// Simulated CProofs of PPE equations with target 1 (one shape per call), randomness drawn per equation in
/// `commit_and_prove`'s order (R rows, S rows, then T).  The openings are not returned: `rand` fields are empty.  Panics
/// when `key` is not the trapdoor of `crs` (any binding CRS) or a target is not 1.
pub fn simulate_ppe<E: Gpu, R: Rng>(equations: &[PPE<E>], crs: &CRS<E>, key: &SimulationKey<E>, rng: &mut R) -> Vec<CProof<E>> {
    if equations.is_empty() { return vec![]; }
    let (m, n) = (equations[0].gamma.len(), equations[0].gamma[0].len());
    let (mut a, mut b, mut g, mut t) = (Vec::new(), Vec::new(), Vec::new(), Vec::new());
    let (mut xr, mut yr, mut pf) = (Vec::new(), Vec::new(), Vec::new());
    for e in equations {
        assert_eq!((e.gamma.len(), e.a_consts.len(), e.b_consts.len()), (m, n, m));
        a.extend(g1s::<E>(&e.a_consts)); b.extend(g2s::<E>(&e.b_consts)); g.extend(fr_matrix::<E>(&e.gamma)); t.push(E::gt(&e.target));
        xr.extend((0..2 * m).map(|_| E::fr(&E::ScalarField::rand(rng))));
        yr.extend((0..2 * n).map(|_| E::fr(&E::ScalarField::rand(rng))));
        pf.extend((0..4).map(|_| E::fr(&E::ScalarField::rand(rng))));
    }
    let k = equations.len();
    let tk = [E::fr(&key.t1), E::fr(&key.t2)];
    let (mut xc, mut yc) = (vec![Com1::<E>::zero().abi(); k * m], vec![Com2::<E>::zero().abi(); k * n]);
    let (mut pi, mut th) = (vec![Com2::<E>::zero().abi(); k * 2], vec![Com1::<E>::zero().abi(); k * 2]);
    with_crs(&crs.abi(), |c| check(c, unsafe {
        gs_simulate_batch(c.raw(), 0, k, m, n, bytes_of(&a).as_ptr(), bytes_of(&b).as_ptr(), g.as_ptr(), bytes_of(&t).as_ptr(),
                          xr.as_ptr(), yr.as_ptr(), pf.as_ptr(), 0, tk.as_ptr(), xc.as_mut_ptr(), yc.as_mut_ptr(), pi.as_mut_ptr(),
                          th.as_mut_ptr())
    }));
    (0..k).map(|i| CProof {
        xcoms: Commit1 { coms: xc[i * m..(i + 1) * m].iter().map(Com1::from_abi).collect(), rand: vec![] },
        ycoms: Commit2 { coms: yc[i * n..(i + 1) * n].iter().map(Com2::from_abi).collect(), rand: vec![] },
        equ_proofs: vec![EquProof { pi: pi[2 * i..2 * i + 2].iter().map(Com2::from_abi).collect(),
                                    theta: th[2 * i..2 * i + 2].iter().map(Com1::from_abi).collect(),
                                    equ_type: EquType::PairingProduct, rand: vec![] }],
    }).collect()
}
