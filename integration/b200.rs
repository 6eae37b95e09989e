// halo2_proofs/src/b200.rs of the patched crate: safe wrappers over b200_sys.rs (generated from include/b200zk.h).
//
// Written against halo2_proofs 1.1.0 @ scroll-tech/halo2 e5ddf67 / halo2curves 0.1.0 @ 112f5b9 (pins:
// /root/reference/Cargo.lock:1886-1888, 1911-1913).  There is no Rust toolchain in the build image of this repository, so this
// file is source for the reference-side integration and is not compiled here; the calling convention it relies on is the one
// the C++ mirror (scroll-prover_b200/halo2_b200.hpp) and the ctypes driver exercise in the test-suite.  See INTEGRATION.md.
#![cfg(feature = "b200")]
use crate::b200_sys as sys;
use halo2curves::bn256::{Fr, G1Affine, G1};
use std::os::raw::{c_int, c_void};

/// One context per process (one process per GPU); created on first use.  `B200ZK_DEVICE` picks the CUDA ordinal.
pub(crate) fn ctx() -> *mut sys::Ctx {
    static CTX: once_cell::sync::Lazy<usize> = once_cell::sync::Lazy::new(|| unsafe {
        let dev: c_int = std::env::var("B200ZK_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        let mut p = std::ptr::null_mut();
        assert_eq!(sys::b200zk_ctx_create(&dev, 1, &mut p), sys::OK, "b200zk: no CUDA device (there is no CPU fallback)");
        p as usize
    });
    *CTX as *mut sys::Ctx
}

/// A failed call becomes the panic the CPU code would have raised (halo2_proofs' arithmetic has no `Result`s).
pub(crate) fn check(rc: i32) {
    if rc != sys::OK {
        let msg = unsafe { std::ffi::CStr::from_ptr(sys::b200zk_last_error(ctx())) }.to_string_lossy().into_owned();
        panic!("b200zk error {rc}: {msg}");
    }
}

fn p<T>(x: &T) -> *const c_void { x as *const T as *const c_void }

/// arithmetic::best_multiexp for C = bn256::G1Affine
pub(crate) fn best_multiexp(coeffs: &[Fr], bases: &[G1Affine]) -> G1 {
    assert_eq!(coeffs.len(), bases.len());
    let mut out = G1::default();
    check(unsafe { sys::b200zk_msm_g1_bases(ctx(), bases.as_ptr() as _, coeffs.as_ptr() as _, coeffs.len() as u64, &mut out as *mut G1 as _) });
    out
}

/// arithmetic::best_fft::<Fr, Fr>
pub(crate) fn best_fft(a: &mut [Fr], omega: Fr, log_n: u32) {
    assert_eq!(a.len(), 1 << log_n);
    check(unsafe { sys::b200zk_ntt_fr(ctx(), a.as_mut_ptr() as _, log_n, p(&omega), 0, sys::COSET_NONE) });
}

/// ParamsKZG::g / g_lagrange resident on the device; registered once, released with the params.
pub(crate) struct DeviceSrs(std::sync::OnceLock<usize>);
impl DeviceSrs {
    pub const fn new() -> Self { DeviceSrs(std::sync::OnceLock::new()) }
    pub fn get_or_register(&self, bases: &[G1Affine], tag: u32) -> *const sys::Srs {
        *self.0.get_or_init(|| {
            let mut h = std::ptr::null_mut();
            check(unsafe { sys::b200zk_srs_register(ctx(), bases.as_ptr() as _, bases.len() as u64, tag, &mut h) });
            h as usize
        }) as *const sys::Srs
    }
}
impl Drop for DeviceSrs {
    fn drop(&mut self) {
        if let Some(h) = self.0.get() { unsafe { sys::b200zk_srs_release(ctx(), *h as *mut sys::Srs) }; }
    }
}

/// ParamsKZG::commit / commit_lagrange (Blind is ignored for KZG, as upstream)
pub(crate) fn commit(srs: *const sys::Srs, values: &[Fr]) -> G1 {
    let mut out = G1::default();
    check(unsafe { sys::b200zk_msm_g1(ctx(), srs, values.as_ptr() as _, values.len() as u64, &mut out as *mut G1 as _) });
    out
}

/// EvaluationDomain::lagrange_to_coeff: ifft with the n^-1 scaling fused
pub(crate) fn lagrange_to_coeff(values: &mut [Fr], k: u32, omega_inv: Fr) {
    check(unsafe { sys::b200zk_ntt_fr(ctx(), values.as_mut_ptr() as _, k, p(&omega_inv), 1, sys::COSET_NONE) });
}
/// EvaluationDomain::coeff_to_extended: distribute_powers_zeta(into_coset), zero extension and the transform in one call
pub(crate) fn coeff_to_extended(coeffs: &[Fr], k: u32, out: &mut [Fr], extended_k: u32, extended_omega: Fr) {
    assert_eq!(coeffs.len(), 1 << k);
    assert_eq!(out.len(), 1 << extended_k);
    check(unsafe { sys::b200zk_ntt_fr_ext(ctx(), coeffs.as_ptr() as _, k, out.as_mut_ptr() as _, extended_k, p(&extended_omega), 0, sys::COSET_PRE) });
}
/// EvaluationDomain::extended_to_coeff (the caller truncates to n * quotient_poly_degree, as upstream)
pub(crate) fn extended_to_coeff(values: &mut [Fr], extended_k: u32, extended_omega_inv: Fr) {
    check(unsafe { sys::b200zk_ntt_fr(ctx(), values.as_mut_ptr() as _, extended_k, p(&extended_omega_inv), 1, sys::COSET_POST) });
}

/// The extended coset by parts (part r = the n points zeta * w_ext^r * w^i): p(zeta * w_ext^part * w^i) for every column, into
/// device buffers of n elements each (the caller keeps them resident, e.g. from b200zk_buf_alloc).
pub(crate) fn coeff_to_extended_parts(columns: &[&[Fr]], k: u32, extended_k: u32, part: u32, out_dev: &[*mut c_void]) {
    assert!(columns.iter().all(|c| c.len() == 1 << k));
    assert_eq!(columns.len(), out_dev.len());
    let ptrs: Vec<*const c_void> = columns.iter().map(|c| c.as_ptr() as *const c_void).collect();
    check(unsafe {
        sys::b200zk_coeff_to_extended_parts(ctx(), ptrs.as_ptr(), ptrs.len() as u32, k, extended_k, part, out_dev.as_ptr())
    });
}
/// divide_by_vanishing_poly (optional) + extended_to_coeff + truncate to n_pieces * n, from the J parts laid out part-major in
/// one device buffer of 2^extended_k elements (consumed); the pieces land in `out_dev` (may be `parts_dev`).
pub(crate) fn extended_parts_to_coeff(parts_dev: *mut c_void, k: u32, extended_k: u32, n_pieces: u32, divide_by_vanishing: bool,
                                      out_dev: *mut c_void) {
    check(unsafe { sys::b200zk_extended_parts_to_coeff(ctx(), parts_dev, k, extended_k, n_pieces, divide_by_vanishing as c_int, out_dev) });
}

pub(crate) fn eval_polynomial(poly: &[Fr], point: Fr) -> Fr {
    let mut out = Fr::zero();
    check(unsafe { sys::b200zk_eval_poly(ctx(), poly.as_ptr() as _, poly.len() as u64, p(&point), &mut out as *mut Fr as _) });
    out
}
pub(crate) fn kate_division(a: &[Fr], b: Fr) -> Vec<Fr> {
    let mut q = vec![Fr::zero(); a.len() - 1];
    check(unsafe { sys::b200zk_kate_division(ctx(), q.as_mut_ptr() as _, a.as_ptr() as _, a.len() as u64, p(&b)) });
    q
}
pub(crate) fn batch_invert(values: &mut [Fr]) {
    check(unsafe { sys::b200zk_batch_invert(ctx(), values.as_mut_ptr() as _, values.len() as u64) });
}

/// One proof phase in one call: every job names its host column, its SRS handle and what to produce
/// (b200zk_run_column_jobs; INTEGRATION.md section 5).  Commitments come back normalised, in job order.
pub(crate) fn run_column_jobs(jobs: &[sys::ColumnJob], k: u32, omega_inv: Fr, extended_omega: Fr, extended_omega_inv: Fr,
                              extended_k: u32) -> Vec<G1> {
    let mut commits = vec![G1::default(); jobs.len()];
    check(unsafe {
        sys::b200zk_run_column_jobs(ctx(), jobs.as_ptr(), jobs.len() as u32, k, p(&omega_inv), p(&extended_omega),
                                    p(&extended_omega_inv), extended_k, commits.as_mut_ptr() as _)
    });
    commits
}

/// The commitments of many columns over one SRS in one batched Pippenger pipeline (b200zk_msm_g1_batch): the advice
/// phase of a wide circuit (the inner proof's several hundred 2^20-row columns).
pub(crate) fn commit_batch(srs: *const sys::Srs, columns: &[&[Fr]]) -> Vec<G1> {
    let n = columns.first().map_or(0, |c| c.len());
    assert!(columns.iter().all(|c| c.len() == n));
    let ptrs: Vec<*const c_void> = columns.iter().map(|c| c.as_ptr() as *const c_void).collect();
    let mut out = vec![G1::default(); columns.len()];
    check(unsafe { sys::b200zk_msm_g1_batch(ctx(), srs, ptrs.as_ptr(), ptrs.len() as u32, n as u64, out.as_mut_ptr() as _) });
    out
}

/// Multi-GPU (one prover process per GPU): join the context-owned NCCL communicator.  Rank 0 obtains `id` with
/// `comm_unique_id()` and ships the 128 bytes to the other processes over the channel they already share.
pub(crate) fn comm_unique_id() -> [u8; 128] {
    let mut id = [0u8; 128];
    assert_eq!(unsafe { sys::b200zk_comm_unique_id(id.as_mut_ptr() as _) }, sys::OK, "b200zk: NCCL not available");
    id
}
pub(crate) fn comm_init(id: &[u8; 128], rank: usize, world: usize) {
    check(unsafe { sys::b200zk_ctx_comm_init(ctx(), id.as_ptr() as _, rank as c_int, world as c_int) });
}
/// best_multiexp over `values` SHARDED BY POINT RANGE across the ranks (collective: every rank calls it with the same
/// polynomial; each uploads only its slice); the same normalised point comes back on every rank.
pub(crate) fn commit_sharded(srs: *const sys::Srs, values: &[Fr], rank: usize, world: usize) -> G1 {
    let (mut first, mut count) = (0u64, 0u64);
    check(unsafe { sys::b200zk_shard_range(values.len() as u64, rank as c_int, world as c_int, &mut first, &mut count) });
    let slice = &values[first as usize..(first + count) as usize];
    let mut out = G1::default();
    check(unsafe { sys::b200zk_msm_g1_sharded(ctx(), srs, slice.as_ptr() as _, values.len() as u64, &mut out as *mut G1 as _) });
    out
}
