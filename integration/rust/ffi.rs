//! Rust binding of liblurk_b200 (C ABI: include/lurk_b200.h).  Hand-written `extern "C"` block + thin safe wrappers, the
//! counterpart of what `pasta-msm` / `grumpkin-msm` are for sppark (SURVEY.md D5).  NOT compiled in the lurk-beta_b200
//! repository (no Rust toolchain in its build image): it is the file a maintainer drops into lurk-beta / Arecibo, next to
//! `build.rs`.  Seams (reference file:line) each wrapper serves are named on the wrapper.
#![allow(non_camel_case_types, dead_code)]
use std::ffi::CStr;
use std::os::raw::{c_char, c_int, c_uint, c_void};

pub const LURK_FIELD_BN254_FR: c_int = 0;
pub const LURK_FIELD_BN254_FQ: c_int = 1;
pub const LURK_FIELD_PALLAS_FQ: c_int = 2;
pub const LURK_FIELD_PALLAS_FP: c_int = 3;
pub const LURK_CURVE_BN254_G1: c_int = 0;
pub const LURK_CURVE_GRUMPKIN: c_int = 1;
pub const LURK_CURVE_PALLAS: c_int = 2;
pub const LURK_CURVE_VESTA: c_int = 3;
pub const LURK_FMT_CANONICAL: c_int = 0;
pub const LURK_FMT_MONTGOMERY: c_int = 1;
pub const LURK_FOLD_BUF_GLUE: c_int = -1;
pub const LURK_FOLD_BUF_X2: c_int = -2;
pub const LURK_FOLD_BUF_RO: c_int = -3;

#[repr(C)]
pub struct lurk_msm_ctx { _private: [u8; 0] }
#[repr(C)]
pub struct lurk_fold_ctx { _private: [u8; 0] }
#[repr(C)]
#[derive(Clone, Copy)]
pub struct lurk_dag_node { pub kind: u8, pub reserved: u8, pub tag: [u16; 4], pub child: [u32; 4] }
#[repr(C)]
pub struct lurk_fold_config {
    pub curve_id: c_int, pub depth: c_int, pub n_w: u64, pub n_x: u64, pub n_rows: u64,
    pub row_ptr: [*const u64; 3], pub col: [*const u32; 3], pub val: [*const u8; 3],
    pub fmt: c_int, pub world: c_int, pub rank: c_int, pub latency_sms: c_int,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct lurk_fold_span { pub first: u64, pub row_elems: u64, pub stride: u64, pub rows: u64 }
#[repr(C)]
pub struct lurk_fold_result {
    pub comm_w: [u8; 96], pub comm_t: [u8; 96], pub r: [u8; 32], pub running_comm_w: [u8; 96], pub running_comm_e: [u8; 96],
    pub ro_hash: [u8; 32], pub status: c_int, pub seq: u64,
}

extern "C" {
    pub fn lurk_last_error() -> *const c_char;
    pub fn lurk_device_count() -> c_int;
    // S1 -- PoseidonCache::hash3/4/6/8 (src/hash.rs:180-203)
    pub fn lurk_poseidon_hash_batch(field_id: c_int, arity: c_int, preimages: *const u8, n: usize, digests: *mut u8) -> c_int;
    pub fn lurk_poseidon_hash_batch_mont(field_id: c_int, arity: c_int, preimages: *const u8, n: usize, digests: *mut u8) -> c_int;
    // S3 -- generate_slots_witnesses (src/lem/multiframe.rs:520-592)
    pub fn lurk_poseidon_witness_block(field_id: c_int, arity: c_int) -> usize;
    pub fn lurk_poseidon_witness_batch(field_id: c_int, arity: c_int, preimages: *const u8, n: usize, blocks: *mut u8, fmt: c_int) -> c_int;
    pub fn lurk_bitdecomp_witness_block(field_id: c_int) -> usize;
    pub fn lurk_bitdecomp_witness_batch(field_id: c_int, values: *const u8, n: usize, blocks: *mut u8, fmt: c_int) -> c_int;
    // S2 -- StoreCore::hydrate_z_cache (src/lem/store_core.rs:256-269)
    pub fn lurk_dag_hash(field_id: c_int, nodes: *const lurk_dag_node, n: usize, atom_digests: *const u8, n_atoms: usize, out: *mut u8) -> c_int;
    // S4 -- Arecibo CommitmentEngineTrait::commit (call sites src/proof/nova.rs:287,292)
    pub fn lurk_msm_ctx_create(curve_id: c_int, bases: *const u8, n: usize, fmt: c_int, out: *mut *mut lurk_msm_ctx) -> c_int;
    pub fn lurk_msm_ctx_precompute(ctx: *mut lurk_msm_ctx) -> c_int;
    pub fn lurk_msm_ctx_run(ctx: *mut lurk_msm_ctx, scalars: *const u8, n: usize, fmt: c_int, out_xyz: *mut u8) -> c_int;
    pub fn lurk_msm_ctx_destroy(ctx: *mut lurk_msm_ctx);
    // S5/S6 -- Proof::prove_recursively (src/proof/nova.rs:260-339, supernova.rs:207-291)
    pub fn lurk_fold_ctx_create(cfg: *const lurk_fold_config, ck_w: *mut lurk_msm_ctx, ck_t: *mut lurk_msm_ctx, out: *mut *mut lurk_fold_ctx) -> c_int;
    pub fn lurk_fold_ctx_destroy(ctx: *mut lurk_fold_ctx);
    pub fn lurk_fold_ctx_add_slot_batch(ctx: *mut lurk_fold_ctx, arity: c_int, count: usize, offsets: *const u64) -> c_int;
    pub fn lurk_fold_ctx_set_spans(ctx: *mut lurk_fold_ctx, n: c_int, spans: *const lurk_fold_span) -> c_int;
    pub fn lurk_fold_ctx_set_ro(ctx: *mut lurk_fold_ctx, n_absorb: c_int, kinds: *const c_int, challenge_bits: c_int) -> c_int;
    pub fn lurk_fold_ctx_host_buffer(ctx: *mut lurk_fold_ctx, b: c_int, which: c_int, ptr: *mut *mut c_void, bytes: *mut usize) -> c_int;
    pub fn lurk_fold_ctx_exchange_handle(ctx: *mut lurk_fold_ctx, handle: *mut u8) -> c_int;
    pub fn lurk_fold_ctx_set_peers(ctx: *mut lurk_fold_ctx, handles: *const u8) -> c_int;
    pub fn lurk_fold_ctx_set_running(ctx: *mut lurk_fold_ctx, w: *const u8, e: *const u8, u: *const u8, x: *const u8, comm_w: *const u8, comm_e: *const u8, fmt: c_int) -> c_int;
    pub fn lurk_fold_ctx_get_running(ctx: *mut lurk_fold_ctx, w: *mut u8, e: *mut u8, u: *mut u8, x: *mut u8, comm_w: *mut u8, comm_e: *mut u8, fmt: c_int) -> c_int;
    pub fn lurk_fold_ctx_stage_a(ctx: *mut lurk_fold_ctx, b: c_int, flags: c_int, fmt: c_int) -> c_int;
    pub fn lurk_fold_ctx_init_running(ctx: *mut lurk_fold_ctx, b: c_int) -> c_int;
    pub fn lurk_fold_ctx_stage_b_launch(ctx: *mut lurk_fold_ctx, b: c_int) -> c_int;
    pub fn lurk_fold_ctx_collect(ctx: *mut lurk_fold_ctx, b: c_int, out: *mut lurk_fold_result, fmt: c_int) -> c_int;
    pub fn lurk_fold_ctx_check_running(ctx: *mut lurk_fold_ctx, bad_rows: *mut u64, comm_w_ok: *mut c_int, comm_e_ok: *mut c_int) -> c_int;
    pub fn lurk_fold_ctx_stats(ctx: *mut lurk_fold_ctx, la: *mut c_uint, lb: *mut c_uint, acc_w_ms: *mut f32, acc_t_ms: *mut f32) -> c_int;
    // N3 -- public_params -> CommitmentKey::setup (src/proof/nova.rs:196-216): from_label (Pedersen engines), powers of tau (HyperKZG)
    pub fn lurk_ck_size(num_cons: usize, num_vars: usize, ck_floor: usize) -> usize;
    pub fn lurk_ck_generate(curve_id: c_int, label: *const u8, label_len: usize, n: usize, fmt: c_int, bases_out: *mut u8) -> c_int;
    pub fn lurk_ck_generate_dev(curve_id: c_int, label: *const u8, label_len: usize, n: usize, d_bases: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn lurk_ck_generate_range_dev(curve_id: c_int, label: *const u8, label_len: usize, first: usize, n: usize, d_bases: *mut c_void, stream: *mut c_void) -> c_int;
    pub fn lurk_ck_powers_dev(curve_id: c_int, g: *const u8, beta: *const u8, n: usize, d_bases: *mut c_void, fmt: c_int, stream: *mut c_void) -> c_int;
    pub fn lurk_msm_ctx_create_dev(curve_id: c_int, d_bases: *const c_void, n: usize, out: *mut *mut lurk_msm_ctx) -> c_int;
    // N4 -- compress (src/proof/nova.rs:341-356): the loops of RelaxedR1CSSNARK::prove / EvaluationEngine::prove; the transcript is the callback
    pub fn lurk_sumcheck_prove_dev(field_id: c_int, kind: c_int, d_polys: *const *mut c_void, num_rounds: c_int, claim: *const u8, challenge: lurk_challenge_fn,
                                   user: *mut c_void, round_evals: *mut u8, challenges: *mut u8, final_evals: *mut u8, fmt: c_int, stream: *mut c_void) -> c_int;
    pub fn lurk_eq_evals_dev(field_id: c_int, tau: *const u8, num_vars: c_int, d_out: *mut c_void, fmt: c_int, stream: *mut c_void) -> c_int;
    pub fn lurk_inner_product_dev(field_id: c_int, d_a: *const c_void, d_b: *const c_void, n: usize, out: *mut u8, fmt: c_int, stream: *mut c_void) -> c_int;
    pub fn lurk_poly_combine_dev(field_id: c_int, n_polys: c_int, d_polys: *const *const c_void, lens: *const usize, coeffs: *const u8, d_out: *mut c_void,
                                 out_len: usize, fmt: c_int, stream: *mut c_void) -> c_int;
    pub fn lurk_ipa_prove_dev(curve_id: c_int, ck: *mut lurk_msm_ctx, ck_c: *const u8, d_a: *mut c_void, d_b: *mut c_void, log_n: c_int, challenge: lurk_challenge_fn,
                              user: *mut c_void, l_out: *mut u8, r_out: *mut u8, a_final: *mut u8, b_final: *mut u8, fmt: c_int, stream: *mut c_void) -> c_int;
    pub fn lurk_hyperkzg_prove_dev(curve_id: c_int, ck: *mut lurk_msm_ctx, d_poly: *const c_void, point: *const u8, num_vars: c_int, challenge: lurk_challenge_fn,
                                   user: *mut c_void, com_out: *mut u8, w_out: *mut u8, v_out: *mut u8, fmt: c_int, stream: *mut c_void) -> c_int;
}
/// `int (*)(void *user, int round, const uint8_t *message, size_t message_len, uint8_t challenge_out[32])`: the Fiat-Shamir transcript stays in
/// Rust.  A closure is passed as `user` and trampolined, e.g. for SumcheckProof::prove_*:
/// `|round, msg| { transcript.absorb(b"p", &UniPoly::from_evals(&elems(msg)).compress()); transcript.squeeze(b"c") }`.
pub type lurk_challenge_fn = unsafe extern "C" fn(user: *mut c_void, round: c_int, message: *const u8, message_len: usize, challenge_out: *mut u8) -> c_int;
pub unsafe extern "C" fn challenge_trampoline<F: FnMut(i32, &[u8]) -> Option<[u8; 32]>>(user: *mut c_void, round: c_int, message: *const u8, len: usize, out: *mut u8) -> c_int {
    let f = &mut *(user as *mut F);
    match f(round, std::slice::from_raw_parts(message, len)) {
        Some(r) => { std::ptr::copy_nonoverlapping(r.as_ptr(), out, 32); 0 }
        None => 1,
    }
}

#[derive(Debug)]
pub struct B200Error { pub code: c_int, pub message: String }
fn check(code: c_int) -> Result<(), B200Error> {
    if code == 0 { return Ok(()); }
    let message = unsafe { CStr::from_ptr(lurk_last_error()) }.to_string_lossy().into_owned();
    Err(B200Error { code, message })
}

/// `PoseidonCache::hashN` for a whole batch: `[F; A]` rows are `repr(C)` `[u64; 4]` Montgomery limbs for pasta_curves
/// (feature `repr-c`, Cargo.toml:42) and halo2curves, so the slices are passed as they are.
pub fn poseidon_hash_batch_mont(field_id: c_int, arity: usize, preimages: &[u8], digests: &mut [u8]) -> Result<(), B200Error> {
    let n = digests.len() / 32;
    assert_eq!(preimages.len(), n * arity * 32);
    check(unsafe { lurk_poseidon_hash_batch_mont(field_id, arity as c_int, preimages.as_ptr(), n, digests.as_mut_ptr()) })
}

/// A device-resident commitment key: what `CommitmentKey<E>` + `commit` become (Arecibo provider; src/proof/nova.rs:196-216).
pub struct MsmCtx(*mut lurk_msm_ctx);
unsafe impl Send for MsmCtx {}
impl MsmCtx {
    pub fn new(curve_id: c_int, bases_affine_mont: &[u8]) -> Result<Self, B200Error> {
        let mut p = std::ptr::null_mut();
        check(unsafe { lurk_msm_ctx_create(curve_id, bases_affine_mont.as_ptr(), bases_affine_mont.len() / 64, LURK_FMT_MONTGOMERY, &mut p) })?;
        check(unsafe { lurk_msm_ctx_precompute(p) })?;
        Ok(Self(p))
    }
    /// `vartime_multiscalar_mul(scalars, bases[..n])` -> x | y | z (z = 1, or all zero for the identity), Montgomery limbs
    pub fn commit(&self, scalars_mont: &[u8]) -> Result<[u8; 96], B200Error> {
        let mut out = [0u8; 96];
        check(unsafe { lurk_msm_ctx_run(self.0, scalars_mont.as_ptr(), scalars_mont.len() / 32, LURK_FMT_MONTGOMERY, out.as_mut_ptr()) })?;
        Ok(out)
    }
    pub fn raw(&self) -> *mut lurk_msm_ctx { self.0 }
}
impl Drop for MsmCtx { fn drop(&mut self) { unsafe { lurk_msm_ctx_destroy(self.0) } } }

/// One running instance on the device (`RecursiveSNARK`'s primary or secondary half; one per circuit index for SuperNova).
pub struct FoldCtx { raw: *mut lurk_fold_ctx, depth: usize, next: usize }
unsafe impl Send for FoldCtx {}
impl FoldCtx {
    /// # Safety: the CSR slices must stay valid for the duration of the call only; `ck` must outlive the context.
    pub unsafe fn new(cfg: &lurk_fold_config, ck_w: &MsmCtx, ck_t: &MsmCtx) -> Result<Self, B200Error> {
        let mut p = std::ptr::null_mut();
        check(lurk_fold_ctx_create(cfg, ck_w.raw(), ck_t.raw(), &mut p))?;
        Ok(Self { raw: p, depth: cfg.depth as usize, next: 0 })
    }
    /// the pinned buffer the witness thread (src/proof/nova.rs:306-318) writes this step's inputs into
    pub fn host_buffer(&mut self, b: usize, which: c_int) -> Result<&mut [u8], B200Error> {
        let (mut p, mut n) = (std::ptr::null_mut(), 0usize);
        check(unsafe { lurk_fold_ctx_host_buffer(self.raw, b as c_int, which, &mut p, &mut n) })?;
        Ok(unsafe { std::slice::from_raw_parts_mut(p as *mut u8, n) })
    }
    pub fn next_buffer(&mut self) -> usize { let b = self.next; self.next = (b + 1) % self.depth; b }
    pub fn stage_a(&mut self, b: usize) -> Result<(), B200Error> { check(unsafe { lurk_fold_ctx_stage_a(self.raw, b as c_int, 0, LURK_FMT_MONTGOMERY) }) }
    pub fn init_running(&mut self, b: usize) -> Result<(), B200Error> { check(unsafe { lurk_fold_ctx_init_running(self.raw, b as c_int) }) }
    pub fn fold(&mut self, b: usize) -> Result<(), B200Error> { check(unsafe { lurk_fold_ctx_stage_b_launch(self.raw, b as c_int) }) }
    pub fn collect(&mut self, b: usize) -> Result<lurk_fold_result, B200Error> {
        let mut r = std::mem::MaybeUninit::<lurk_fold_result>::zeroed();
        check(unsafe { lurk_fold_ctx_collect(self.raw, b as c_int, r.as_mut_ptr(), LURK_FMT_MONTGOMERY) })?;
        Ok(unsafe { r.assume_init() })
    }
}
impl Drop for FoldCtx { fn drop(&mut self) { unsafe { lurk_fold_ctx_destroy(self.raw) } } }
