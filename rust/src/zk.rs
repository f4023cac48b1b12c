//! Not in the reference: zero-knowledge proofs of PPEs whose target is given as K public pairs,
//! sum_k e(P_k, Q_k) (Groth & Sahai, EUROCRYPT 2008).  The statement is augmented to a target-1 PPE' over (X | Z) with
//! constants (B | -Q) and K equations Z_k - delta P_k = O whose delta has the fixed commitment W2 (include/gs_b200.h,
//! `gs_zk_ppe_prove_batch`).  `prove` makes real proofs, `simulate` makes proofs for any target pairs with the hiding
//! CRS's trapdoor, `verify` checks both, `rerandomize` refreshes either without witness or trapdoor; real and simulated
//! proofs are identically distributed under a hiding CRS.
use crate::data_structures::{Com1, Com2};
use crate::ffi::*;
use crate::generator::CRS;
use crate::prover::{Commit1, Commit2, EquProof};
use crate::simulator::SimulationKey;
use crate::statement::EquType;
use ark_ff::{UniformRand, Zero};
use ark_std::rand::Rng;

/// sum_j e(A_j, Y_j) + sum_i e(X_i, B_i) + sum_ij gamma_ij e(X_i, Y_j) = sum_k e(P_k, Q_k)
pub struct ZkPPE<E: Gpu> {
    pub a_consts: Vec<E::G1Affine>,
    pub b_consts: Vec<E::G2Affine>,
    pub gamma: Vec<Vec<E::ScalarField>>,
    pub target_pairs: Vec<(E::G1Affine, E::G2Affine)>,
}

/// xcoms: m + K (X, then Z); ppe: the proof of PPE'; lin: the K proofs of Z_k - delta P_k = O
pub struct ZkPPEProof<E: Gpu> { pub xcoms: Commit1<E>, pub ycoms: Commit2<E>, pub ppe: EquProof<E>, pub lin: Vec<EquProof<E>> }

impl<E: Gpu> ZkPPE<E> {
    fn shape(&self) -> (usize, usize, usize) {
        assert_eq!(self.gamma.len(), self.b_consts.len());
        assert!(self.gamma.iter().all(|r| r.len() == self.a_consts.len()));
        (self.b_consts.len(), self.a_consts.len(), self.target_pairs.len())
    }

    fn statement(&self) -> (Vec<GsG1>, Vec<GsG2>, Vec<GsFr>, Vec<GsG1>, Vec<GsG2>) {
        let tp: Vec<E::G1Affine> = self.target_pairs.iter().map(|p| p.0).collect();
        let tq: Vec<E::G2Affine> = self.target_pairs.iter().map(|p| p.1).collect();
        (g1s::<E>(&self.a_consts), g2s::<E>(&self.b_consts), fr_matrix::<E>(&self.gamma), g1s::<E>(&tp), g2s::<E>(&tq))
    }

    /// randomness in the engine's order: R ((m + K) x 2), S (n x 2), T (2 x 2), T_1..T_K (1 x 2)
    fn draws<R: Rng>(&self, rng: &mut R) -> Vec<Vec<Vec<E::ScalarField>>> {
        let (m, n, k) = self.shape();
        [m + k, n, 2, k].iter().map(|&rows| (0..rows).map(|_| (0..2).map(|_| E::ScalarField::rand(rng)).collect()).collect()).collect()
    }

    fn proof(&self, d: Vec<Vec<Vec<E::ScalarField>>>, out: (Vec<GsCom1>, Vec<GsCom2>, Vec<GsCom2>, Vec<GsCom1>, Vec<GsCom2>, Vec<GsCom1>),
             keep_rand: bool) -> ZkPPEProof<E> {
        let (xc, yc, pi, th, lpi, lth) = out;
        let r = |i: usize| if keep_rand { d[i].clone() } else { vec![] };
        ZkPPEProof {
            xcoms: Commit1 { coms: xc.iter().map(Com1::from_abi).collect(), rand: r(0) },
            ycoms: Commit2 { coms: yc.iter().map(Com2::from_abi).collect(), rand: r(1) },
            ppe: EquProof { pi: pi.iter().map(Com2::from_abi).collect(), theta: th.iter().map(Com1::from_abi).collect(),
                            equ_type: EquType::PairingProduct, rand: r(2) },
            lin: (0..lth.len()).map(|k| EquProof { pi: lpi[2 * k..2 * k + 2].iter().map(Com2::from_abi).collect(),
                                                   theta: vec![Com1::from_abi(&lth[k])], equ_type: EquType::MultiScalarG1,
                                                   rand: if keep_rand { vec![d[3][k].clone()] } else { vec![] } }).collect(),
        }
    }

    fn outs(&self) -> (Vec<GsCom1>, Vec<GsCom2>, Vec<GsCom2>, Vec<GsCom1>, Vec<GsCom2>, Vec<GsCom1>) {
        let (m, n, k) = self.shape();
        (vec![Com1::<E>::zero().abi(); m + k], vec![Com2::<E>::zero().abi(); n], vec![Com2::<E>::zero().abi(); 2],
         vec![Com1::<E>::zero().abi(); 2], vec![Com2::<E>::zero().abi(); 2 * k], vec![Com1::<E>::zero().abi(); k])
    }

    /// A zero-knowledge proof from witnesses xvars (m) and yvars (n) that satisfy the statement.
    pub fn prove<R: Rng>(&self, xvars: &[E::G1Affine], yvars: &[E::G2Affine], crs: &CRS<E>, rng: &mut R) -> ZkPPEProof<E> {
        let (m, n, k) = self.shape();
        assert_eq!((xvars.len(), yvars.len()), (m, n));
        let d = self.draws(rng);
        let (a, b, g, tp, tq) = self.statement();
        let (x, y) = (g1s::<E>(xvars), g2s::<E>(yvars));
        let r: Vec<Vec<GsFr>> = d.iter().map(|mat| fr_matrix::<E>(mat)).collect();
        let mut o = self.outs();
        with_crs(&crs.abi(), |c| check(c, unsafe {
            gs_zk_ppe_prove_batch(c.raw(), 1, m, n, k, a.as_ptr(), b.as_ptr(), g.as_ptr(), tp.as_ptr(), tq.as_ptr(), x.as_ptr(), y.as_ptr(),
                                  r[0].as_ptr(), r[1].as_ptr(), r[2].as_ptr(), r[3].as_ptr(), o.0.as_mut_ptr(), o.1.as_mut_ptr(),
                                  o.2.as_mut_ptr(), o.3.as_mut_ptr(), o.4.as_mut_ptr(), o.5.as_mut_ptr())
        }));
        self.proof(d, o, true)
    }

    /// A proof that verifies under the hiding CRS `crs` for any target pairs, made with its trapdoor; panics when `key`
    /// is not the trapdoor of `crs` (any binding CRS).  Draws as `prove`; the openings are not returned.
    pub fn simulate<R: Rng>(&self, crs: &CRS<E>, key: &SimulationKey<E>, rng: &mut R) -> ZkPPEProof<E> {
        let (m, n, k) = self.shape();
        let d = self.draws(rng);
        let (a, b, g, tp, tq) = self.statement();
        let r: Vec<Vec<GsFr>> = d.iter().map(|mat| fr_matrix::<E>(mat)).collect();
        let tk = [E::fr(&key.t1), E::fr(&key.t2)];
        let mut o = self.outs();
        with_crs(&crs.abi(), |c| check(c, unsafe {
            gs_zk_ppe_simulate_batch(c.raw(), 1, m, n, k, a.as_ptr(), b.as_ptr(), g.as_ptr(), tp.as_ptr(), tq.as_ptr(), r[0].as_ptr(),
                                     r[1].as_ptr(), r[2].as_ptr(), r[3].as_ptr(), tk.as_ptr(), o.0.as_mut_ptr(), o.1.as_mut_ptr(),
                                     o.2.as_mut_ptr(), o.3.as_mut_ptr(), o.4.as_mut_ptr(), o.5.as_mut_ptr())
        }));
        self.proof(d, o, false)
    }

    /// Not in the reference: a fresh-looking proof of the same statement from `proof` alone, real or simulated, without
    /// witness or trapdoor (Belenkiy et al., CRYPTO 2009; gs_zk_ppe_rerandomize_batch).  Fresh randomness is drawn as for
    /// `prove`; the openings are not returned.  The input is not checked: a proof that fails `verify` still fails.
    pub fn rerandomize<R: Rng>(&self, proof: &ZkPPEProof<E>, crs: &CRS<E>, rng: &mut R) -> ZkPPEProof<E> {
        let (m, n, k) = self.shape();
        assert_eq!((proof.xcoms.coms.len(), proof.ycoms.coms.len(), proof.lin.len()), (m + k, n, k));
        let (a, b, g, _, tq) = self.statement();
        let (xc, yc, pi, th, lpi, lth) = Self::proof_abi(proof);
        assert_eq!((pi.len(), th.len(), lpi.len(), lth.len()), (2, 2, 2 * k, k));
        let d = self.draws(rng);
        let r: Vec<Vec<GsFr>> = d.iter().map(|mat| fr_matrix::<E>(mat)).collect();
        let mut o = self.outs();
        with_crs(&crs.abi(), |c| check(c, unsafe {
            gs_zk_ppe_rerandomize_batch(c.raw(), 1, m, n, k, a.as_ptr(), b.as_ptr(), g.as_ptr(), tq.as_ptr(), xc.as_ptr(),
                                        yc.as_ptr(), pi.as_ptr(), th.as_ptr(), lpi.as_ptr(), lth.as_ptr(), r[0].as_ptr(),
                                        r[1].as_ptr(), r[2].as_ptr(), r[3].as_ptr(), o.0.as_mut_ptr(), o.1.as_mut_ptr(),
                                        o.2.as_mut_ptr(), o.3.as_mut_ptr(), o.4.as_mut_ptr(), o.5.as_mut_ptr())
        }));
        self.proof(d, o, false)
    }

    fn proof_abi(proof: &ZkPPEProof<E>) -> (Vec<GsCom1>, Vec<GsCom2>, Vec<GsCom2>, Vec<GsCom1>, Vec<GsCom2>, Vec<GsCom1>) {
        (proof.xcoms.coms.iter().map(|c| c.abi()).collect(), proof.ycoms.coms.iter().map(|c| c.abi()).collect(),
         proof.ppe.pi.iter().map(|c| c.abi()).collect(), proof.ppe.theta.iter().map(|c| c.abi()).collect(),
         proof.lin.iter().flat_map(|e| e.pi.iter().map(|c| c.abi())).collect(),
         proof.lin.iter().flat_map(|e| e.theta.iter().map(|c| c.abi())).collect())
    }

    /// PPE' and every Z_k - delta P_k = O verify, delta's commitment being W2 of `crs`.
    pub fn verify(&self, proof: &ZkPPEProof<E>, crs: &CRS<E>) -> bool {
        self.verify_with(proof, crs, None)
    }

    /// Not in the reference: the verdict of `verify` at close to the cost of one equation (gs_zk_ppe_verify_each_rand):
    /// PPE' and the K equations are folded, each with its own weights from `rng` (a cryptographic RNG the prover cannot
    /// predict), into one pairing product and ONE final exponentiation.  A bad proof is accepted with probability <= 2^-62.
    pub fn verify_each_randomized(&self, proof: &ZkPPEProof<E>, crs: &CRS<E>, rng: &mut dyn ark_std::rand::RngCore) -> bool {
        let rho: Vec<u64> = (0..2 * (1 + self.target_pairs.len()) + 1).map(|_| rng.next_u64()).collect();
        self.verify_with(proof, crs, Some(&rho))
    }

    fn verify_with(&self, proof: &ZkPPEProof<E>, crs: &CRS<E>, rho: Option<&[u64]>) -> bool {
        let (m, n, k) = self.shape();
        assert_eq!((proof.xcoms.coms.len(), proof.ycoms.coms.len(), proof.lin.len()), (m + k, n, k));
        let (a, b, g, tp, tq) = self.statement();
        let (xc, yc, pi, th, lpi, lth) = Self::proof_abi(proof);
        assert_eq!((pi.len(), th.len(), lpi.len(), lth.len()), (2, 2, 2 * k, k));
        let mut ok = [0u8];
        with_crs(&crs.abi(), |c| check(c, unsafe {
            match rho {
                None => gs_zk_ppe_verify_batch(c.raw(), 1, m, n, k, a.as_ptr(), b.as_ptr(), g.as_ptr(), tp.as_ptr(), tq.as_ptr(),
                                               xc.as_ptr(), yc.as_ptr(), pi.as_ptr(), th.as_ptr(), lpi.as_ptr(), lth.as_ptr(),
                                               ok.as_mut_ptr()),
                Some(r) => gs_zk_ppe_verify_each_rand(c.raw(), 1, m, n, k, a.as_ptr(), b.as_ptr(), g.as_ptr(), tp.as_ptr(),
                                                      tq.as_ptr(), xc.as_ptr(), yc.as_ptr(), pi.as_ptr(), th.as_ptr(), lpi.as_ptr(),
                                                      lth.as_ptr(), r.as_ptr(), ok.as_mut_ptr()),
            }
        }));
        ok[0] == 1
    }
}
