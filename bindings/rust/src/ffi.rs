//! Raw declarations, one for one with include/b2m.h.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_uint, c_ulonglong, c_void};

#[repr(C)]
pub struct b2m_ctx {
    _p: [u8; 0],
}
#[repr(C)]
pub struct b2m_srs {
    _p: [u8; 0],
}
#[repr(C)]
pub struct b2m_index {
    _p: [u8; 0],
}
#[repr(C)]
pub struct b2m_ck {
    _p: [u8; 0],
}
#[repr(C)]
pub struct b2m_verifier {
    _p: [u8; 0],
}
#[repr(C)]
pub struct b2m_matrix {
    pub row_ptr: *const u64,
    pub col: *const u64,
    pub coeff: *const u64,
}
/// `b2m_rng` (include/b2m.h): a ChaCha stream position (kind = 8 / 12 / 20) or, with kind = B2M_RNG_CALLBACK, any `RngCore`
/// reached through `next_u64(state)`.
#[repr(C)]
#[derive(Clone, Copy)]
pub struct b2m_rng {
    pub kind: c_int,
    pub key: [u8; 32],
    pub word_pos: u64,
    pub next_u64: Option<unsafe extern "C" fn(state: *mut c_void) -> u64>,
    pub state: *mut c_void,
}
pub const B2M_RNG_CALLBACK: c_int = 1;

pub const B2M_OK: c_int = 0;
pub const B2M_ERR_INVALID_ARG: c_int = 1;
pub const B2M_ERR_INDEX_TOO_LARGE: c_int = 2;
pub const B2M_ERR_INSTANCE_MISMATCH: c_int = 3;
pub const B2M_ERR_INVALID_PUBLIC_INPUT_LEN: c_int = 4;
pub const B2M_ERR_NON_SQUARE: c_int = 5;
pub const B2M_ERR_DEGREE_TOO_LARGE: c_int = 6;
pub const B2M_ERR_MISSING_RNG: c_int = 7;
pub const B2M_ERR_CUDA: c_int = 8;
pub const B2M_ERR_NCCL: c_int = 9;
pub const B2M_ERR_UNSUPPORTED: c_int = 10;
pub const B2M_CURVE_BLS12_381: c_int = 0;
pub const B2M_CURVE_BN254: c_int = 1;
pub const B2M_PC_MARLIN_KZG10: c_int = 0;
pub const B2M_PC_SONIC_KZG10: c_int = 1;

extern "C" {
    pub fn b2m_last_error() -> *const c_char;
    pub fn b2m_version() -> *const c_char;
    pub fn b2m_ctx_create(device: c_int, out: *mut *mut b2m_ctx) -> c_int;
    pub fn b2m_ctx_destroy(ctx: *mut b2m_ctx);
    pub fn b2m_ctx_launches(ctx: *const b2m_ctx) -> c_ulonglong;
    pub fn b2m_comm_unique_id(id: *mut u8, cap: usize) -> c_int;
    pub fn b2m_ctx_attach_comm(ctx: *mut b2m_ctx, id: *const u8, id_len: usize, rank: c_int, world: c_int) -> c_int;
    pub fn b2m_ntt(ctx: *mut b2m_ctx, curve: c_int, data: *mut u64, log_n: c_uint, inverse: c_int, coset: c_int) -> c_int;
    pub fn b2m_msm_g1(ctx: *mut b2m_ctx, curve: c_int, bases_xy: *const u64, scalars: *const u64, n: usize, out_xy: *mut u64,
                      out_is_inf: *mut c_int) -> c_int;
    pub fn b2m_srs_create(ctx: *mut b2m_ctx, curve: c_int, powers_of_g: *const u64, n_g: usize, powers_of_gamma_g: *const u64,
                          gamma_indices: *const u64, n_gamma: usize, window_bits: c_int, out: *mut *mut b2m_srs) -> c_int;
    pub fn b2m_srs_destroy(srs: *mut b2m_srs);
    pub fn b2m_srs_size(srs: *const b2m_srs) -> usize;
    pub fn b2m_srs_msm(srs: *mut b2m_srs, base_off: usize, scalars: *const u64, n: usize, out_xy: *mut u64, out_is_inf: *mut c_int) -> c_int;
    pub fn b2m_pc_commit(srs: *mut b2m_srs, pc_variant: c_int, n_polys: usize, coeffs: *const *const u64, n_coeffs: *const usize,
                         degree_bounds: *const i64, hiding_bounds: *const i64, rng: *mut b2m_rng, out_comm_xy: *mut u64,
                         out_shifted_xy: *mut u64, out_rand: *mut u64, out_shifted_rand: *mut u64, rand_stride: usize) -> c_int;
    pub fn b2m_pc_open(srs: *mut b2m_srs, pc_variant: c_int, n_polys: usize, coeffs: *const *const u64, n_coeffs: *const usize,
                       degree_bounds: *const i64, rands: *const u64, shifted_rands: *const u64, rand_stride: usize,
                       max_degree_bound: i64, point: *const u64, opening_challenge: *const u64, out_w_xy: *mut u64,
                       out_has_random_v: *mut c_int, out_random_v: *mut u64) -> c_int;
    pub fn b2m_g1_powers(ctx: *mut b2m_ctx, curve: c_int, g_xy: *const u64, beta: *const u64, n: usize, out_powers_xy: *mut u64) -> c_int;
    pub fn b2m_fixed_base_msm(ctx: *mut b2m_ctx, curve: c_int, g_xy: *const u64, scalars: *const u64, n: usize, out_xy: *mut u64) -> c_int;
    pub fn b2m_trim(srs: *mut b2m_srs, pc_variant: c_int, supported_degree: usize, supported_hiding_bound: usize,
                    enforced_degree_bounds: *const u64, n_bounds: usize, out: *mut *mut b2m_ck) -> c_int;
    pub fn b2m_ck_destroy(ck: *mut b2m_ck);
    pub fn b2m_ck_supported_degree(ck: *const b2m_ck) -> usize;
    pub fn b2m_ck_shift_power(ck: *const b2m_ck, bound: u64, out_xy: *mut u64) -> c_int;
    pub fn b2m_ck_commit(ck: *mut b2m_ck, n_polys: usize, coeffs: *const *const u64, n_coeffs: *const usize, degree_bounds: *const i64,
                         hiding_bounds: *const i64, rng: *mut b2m_rng, out_comm_xy: *mut u64, out_shifted_xy: *mut u64, out_rand: *mut u64,
                         out_shifted_rand: *mut u64, rand_stride: usize) -> c_int;
    pub fn b2m_ck_open_combinations(ck: *mut b2m_ck, n_polys: usize, coeffs: *const *const u64, n_coeffs: *const usize,
                                    degree_bounds: *const i64, hiding: *const c_int, rands: *const u64, shifted_rands: *const u64,
                                    rand_stride: usize, n_lcs: usize, lc_term_off: *const usize, lc_poly: *const i64, lc_coeff: *const u64,
                                    n_queries: usize, query_lc: *const usize, query_point: *const usize, n_points: usize,
                                    points: *const u64, opening_challenge: *const u64, out_w_xy: *mut u64, out_has_random_v: *mut c_int,
                                    out_random_v: *mut u64) -> c_int;
    pub fn b2m_index_create(srs: *mut b2m_srs, pc_variant: c_int, num_constraints: usize, num_variables: usize,
                            num_instance_variables: usize, a: *const b2m_matrix, b: *const b2m_matrix, c: *const b2m_matrix,
                            out: *mut *mut b2m_index) -> c_int;
    pub fn b2m_index_destroy(idx: *mut b2m_index);
    pub fn b2m_index_vk_bytes(idx: *const b2m_index, out: *mut u8, cap: usize, len: *mut usize) -> c_int;
    pub fn b2m_index_comms(idx: *const b2m_index, out_xy: *mut u64) -> c_int;
    pub fn b2m_prove(idx: *mut b2m_index, formatted_input: *const u64, n_input: usize, witness: *const u64, n_witness: usize,
                     zk_rng: *mut b2m_rng, proof: *mut u8, cap: usize, proof_len: *mut usize) -> c_int;
    pub fn b2m_verifier_create(ctx: *mut b2m_ctx, curve: c_int, pc_variant: c_int, vk_tobytes: *const u8, vk_len: usize, g: *const u8,
                               gamma_g: *const u8, h: *const u8, beta_h: *const u8, max_degree: usize, n_bounds: usize,
                               bounds: *const u64, bound_points: *const u8, out: *mut *mut b2m_verifier) -> c_int;
    pub fn b2m_verifier_destroy(ver: *mut b2m_verifier);
    pub fn b2m_verify(ver: *mut b2m_verifier, n_proofs: usize, public_inputs: *const *const u64, n_inputs: *const usize,
                      proofs: *const *const u8, proof_lens: *const usize, rng: *mut b2m_rng, verdicts: *mut c_int) -> c_int;
    pub fn b2m_verify_timings(ver: *const b2m_verifier, json: *mut c_char, cap: usize) -> c_int;
}
