//! groth-sahai-rs with its hot path on a B200: the module tree and public signatures of the reference
//! (`src/lib.rs:1-9`, `src/prover/mod.rs:1-5`), every arithmetic body replaced by a call into
//! `libgs_b200.so` (`ffi.rs`, one `extern "C"` line per symbol of `include/gs_b200.h`).
//!
//! Differences a user can observe:
//! * every generic `E: Pairing` additionally needs `E: Gpu` (`ffi::Gpu`), implemented for
//!   `ark_bls12_381::Bls12_381` only -- another curve is a compile error instead of a CPU fallback;
//! * randomness is still drawn from the caller's `Rng` in the reference's order (commit rows, then T) on the host;
//! * dimension errors are the same panics (the C ABI's `GS_EDIM` is re-raised by `ffi::check`).
#![allow(non_snake_case)]
pub mod data_structures;
pub mod extractor;
pub mod ffi;
pub mod generator;
pub mod prover;
pub mod statement;
pub mod verifier;

pub use crate::generator::{AbstractCrs, CRS};
pub use crate::statement::*;
