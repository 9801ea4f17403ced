//! `extern "C"` declarations of include/qfall_b200.h, one for one (checked by
//! tests/test_host_logic.py::test_rust_shim_matches_header: same names, same parameter counts).
#![allow(non_camel_case_types, clippy::too_many_arguments)]
use core::ffi::{c_char, c_void};

pub const QF_OK: i32 = 0;
pub const QF_ERR_INVALID: i32 = 1;
pub const QF_ERR_CUDA: i32 = 2;
pub const QF_ERR_NOT_IN_DOMAIN: i32 = 3;
pub const QF_ERR_NO_KEY: i32 = 4;
pub const QF_ERR_UNSUPPORTED: i32 = 5;
pub const QF_ERR_NUMERIC: i32 = 6;

pub const QF_PSF_GPV: i32 = 0;
pub const QF_PSF_PERTURBATION: i32 = 1;
pub const QF_PSF_GPV_RING: i32 = 2;

#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct qf_params {
    pub kind: i32,
    pub n: i64,
    pub k: i64,
    pub m_bar: i64,
    pub base: i64,
    pub q: u64,
    pub s: f64,
    pub r: f64,
    pub norm_bound: u64,
}

#[repr(C)]
pub struct qf_ctx {
    _private: [u8; 0],
}

extern "C" {
    pub fn qf_ctx_create(params: *const qf_params, device: i32, out: *mut *mut qf_ctx) -> i32;
    pub fn qf_ctx_destroy(ctx: *mut qf_ctx);
    pub fn qf_last_error(ctx: *const qf_ctx) -> *const c_char;
    pub fn qf_set_stream(ctx: *mut qf_ctx, cuda_stream: *mut c_void) -> i32;
    pub fn qf_set_chunk(ctx: *mut qf_ctx, targets_per_chunk: i64) -> i32;
    pub fn qf_synchronize(ctx: *mut qf_ctx) -> i32;
    pub fn qf_launch_count(ctx: *const qf_ctx) -> u64;
    pub fn qf_profile(ctx: *mut qf_ctx, enable: i32) -> i32;
    pub fn qf_profile_read(ctx: *mut qf_ctx, gemm_ms: *mut f64, gemm_flops: *mut f64, gemm_launches: *mut u64, i8_ms: *mut f64, i8_ops: *mut f64, i8_issued_ops: *mut f64, i8_launches: *mut u64) -> i32;

    pub fn qf_set_a(ctx: *mut qf_ctx, a: *const i64) -> i32;
    pub fn qf_set_trapdoor_perturbation(ctx: *mut qf_ctx, r: *const i8, sqrt_sigma_2: *const f64, s_block: *const i64, s_block_gso: *const f64) -> i32;
    pub fn qf_set_tag(ctx: *mut qf_ctx, tag: *const i64, a_out: *mut i64) -> i32;
    pub fn qf_gpv_set_tag(ctx: *mut qf_ctx, tag: *const i64, a_out: *mut i64, s_out: *mut i64) -> i32;
    pub fn qf_set_tag_table(ctx: *mut qf_ctx, tags: *const i64, ntags: i64) -> i32;
    pub fn qf_set_f_a_tags(ctx: *mut qf_ctx, tags: *const i64, ntags: i64, h0: *const i64) -> i32;
    pub fn qf_set_tag_table_poly(ctx: *mut qf_ctx, f: *const i64, tags: *const i64, ntags: i64) -> i32;
    pub fn qf_set_f_a_tags_poly(ctx: *mut qf_ctx, f: *const i64, tags: *const i64, ntags: i64, h0: *const i64) -> i32;
    pub fn qf_gen_short_basis(ctx: *mut qf_ctx, r: *const i8, s_out: *mut i64) -> i32;
    pub fn qf_gen_short_basis_tagged(ctx: *mut qf_ctx, r: *const i8, tag: *const i64, s_out: *mut i64) -> i32;
    pub fn qf_compute_sqrt_sigma_2(ctx: *mut qf_ctx, r: *const i8, sigma: *const f64, sqrt_sigma_2_out: *mut f64) -> i32;
    pub fn qf_set_trapdoor_gpv(ctx: *mut qf_ctx, s: *const i64, s_gso: *const f64) -> i32;
    pub fn qf_gso(ctx: *mut qf_ctx, s: *const i64, gso_out: *mut f64) -> i32;
    pub fn qf_ring_gen_short_basis(ctx: *mut qf_ctx, r: *const i32, e: *const i32, s_out: *mut i64) -> i32;
    pub fn qf_ring_set_a(ctx: *mut qf_ctx, a: *const i64) -> i32;

    pub fn qf_trap_gen_from(ctx: *mut qf_ctx, a_bar: *const i64, r: *const i8, tag: *const i64, a_out: *mut i64) -> i32;
    pub fn qf_trap_gen(ctx: *mut qf_ctx, seed: u64, a_out: *mut i64, r_out: *mut i8) -> i32;
    pub fn qf_ring_trap_gen_from(ctx: *mut qf_ctx, a_bar: *const i64, r: *const i32, e: *const i32, a_out: *mut i64) -> i32;

    pub fn qf_f_a(ctx: *mut qf_ctx, sigma: *const i32, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_f_a_dev(ctx: *mut qf_ctx, sigma: *const i32, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_check_domain(ctx: *mut qf_ctx, sigma: *const i32, batch: i64, in_domain: *mut u8) -> i32;
    pub fn qf_f_a_tagged(ctx: *mut qf_ctx, sigma: *const i32, tag_idx: *const i32, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_f_a_tagged_dev(ctx: *mut qf_ctx, sigma: *const i32, tag_idx: *const i32, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_ring_set_key_table(ctx: *mut qf_ctx, keys: *const i64, nkeys: i64) -> i32;
    pub fn qf_ring_f_a_keyed(ctx: *mut qf_ctx, sigma: *const i32, key_idx: *const i32, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_ring_f_a_keyed_dev(ctx: *mut qf_ctx, sigma: *const i32, key_idx: *const i32, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_ring_f_a_keyed_packed(ctx: *mut qf_ctx, packed: *const u8, key_idx: *const i32, batch: i64, k: i32, slot_bytes: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_ring_f_a_keyed_packed_dev(ctx: *mut qf_ctx, packed: *const u8, key_idx: *const i32, batch: i64, k: i32, slot_bytes: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_ring_trap_gen_batch_from(ctx: *mut qf_ctx, count: i64, a_bar: *const i64, r: *const i32, e: *const i32, a_out: *mut i64) -> i32;
    pub fn qf_samp_d(ctx: *mut qf_ctx, batch: i64, seed: u64, first_index: u64, out: *mut i32) -> i32;
    pub fn qf_samp_d_dev(ctx: *mut qf_ctx, batch: i64, seed: u64, first_index: u64, out: *mut i32) -> i32;
    pub fn qf_samp_p(ctx: *mut qf_ctx, u: *const i64, batch: i64, seed: u64, first_index: u64, e_out: *mut i32) -> i32;
    pub fn qf_samp_p_dev(ctx: *mut qf_ctx, u: *const i64, batch: i64, seed: u64, first_index: u64, e_out: *mut i32) -> i32;

    pub fn qf_samp_p_tagged(ctx: *mut qf_ctx, u: *const i64, tag_idx: *const i32, batch: i64, seed: u64, first_index: u64, e_out: *mut i32) -> i32;
    pub fn qf_samp_p_tagged_dev(ctx: *mut qf_ctx, u: *const i64, tag_idx: *const i32, batch: i64, seed: u64, first_index: u64, e_out: *mut i32) -> i32;
    pub fn qf_samp_p_offline(ctx: *mut qf_ctx, count: i64, seed: u64, first_index: u64) -> i32;
    pub fn qf_samp_p_pool_info(ctx: *const qf_ctx, remaining: *mut i64, next_index: *mut u64) -> i32;
    pub fn qf_samp_p_online(ctx: *mut qf_ctx, u: *const i64, tag_idx: *const i32, batch: i64, e_out: *mut i32, first_index_out: *mut u64) -> i32;
    pub fn qf_samp_p_online_dev(ctx: *mut qf_ctx, u: *const i64, tag_idx: *const i32, batch: i64, e_out: *mut i32, first_index_out: *mut u64) -> i32;
    pub fn qf_samp_p_i16(ctx: *mut qf_ctx, u: *const i64, batch: i64, seed: u64, first_index: u64, e_out: *mut i16) -> i32;
    pub fn qf_f_a_i16(ctx: *mut qf_ctx, sigma: *const i16, batch: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_narrow_i32_i16_dev(input: *const i32, out: *mut i16, count: usize, overflow: *mut i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_domain_code_params(ctx: *mut qf_ctx, k: *mut i32, slot_bytes: *mut i64) -> i32;
    pub fn qf_samp_p_packed(ctx: *mut qf_ctx, u: *const i64, tag_idx: *const i32, batch: i64, seed: u64, first_index: u64, k: i32, slot_bytes: i64, out: *mut u8, nbytes: *mut i32) -> i32;
    pub fn qf_f_a_packed(ctx: *mut qf_ctx, packed: *const u8, tag_idx: *const i32, batch: i64, k: i32, slot_bytes: i64, u_out: *mut i64, in_domain: *mut u8) -> i32;
    pub fn qf_domain_encode_dev(input: *const i32, rows: i64, dim: i64, k: i32, slot_bytes: i64, out: *mut u8, nbytes: *mut i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_domain_decode_dev(input: *const u8, rows: i64, dim: i64, k: i32, slot_bytes: i64, out: *mut i32, ok: *mut u8, cuda_stream: *mut c_void) -> i32;
    pub fn qf_randomized_nearest_plane_gadget(ctx: *mut qf_ctx, v: *const i64, batch: i64, seed: u64, first_index: u64, z_out: *mut i32) -> i32;

    pub fn qf_compress_u16(input: *const u16, out: *mut u16, count: usize, q: u32, d: u32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_decompress_u16(input: *const u16, out: *mut u16, count: usize, q: u32, d: u32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_compress_i64(input: *const i64, out: *mut i64, count: usize, q: u64, d: u32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_decompress_i64(input: *const i64, out: *mut i64, count: usize, q: u64, d: u32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_compress_encode_u16(input: *const u16, out: *mut u8, npoly: usize, q: u32, d: u32, compress: i32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_decode_decompress_u16(input: *const u8, out: *mut u16, npoly: usize, q: u32, d: u32, decompress: i32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;

    pub fn qf_encode_digits(digits: *const u8, coeffs: *mut c_void, count: usize, q: u64, base: u32, coeff_bytes: i32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_decode_digits(coeffs: *const c_void, digits: *mut u8, count: usize, q: u64, base: u32, coeff_bytes: i32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_encode_bits_u16(msg: *const u8, coeffs: *mut u16, nbytes: usize, q: u32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_decode_bits_u16(coeffs: *const u16, msg: *mut u8, nbytes: usize, q: u32, device_ptrs: i32, cuda_stream: *mut c_void) -> i32;
    pub fn qf_sample_z(centers: *const f64, count: usize, s: f64, seed: u64, out: *mut i64) -> i32;
    pub fn qf_debug_gemm_i8(x: *const i64, w: *const i64, w_signed: i32, lx: i32, lw: i32, b: i64, n: i64, k: i64, q: u64, out: *mut i64) -> i32;
    pub fn qf_probe_i8_peak(device: i32, b: i64, n: i64, k: i64, iters: i32, sustain_ms: f64, best_tops: *mut f64, sustained_tops: *mut f64, pipe_tops: *mut f64) -> i32;
    pub fn qf_fill_uniform_modq_dev(out: *mut i64, count: usize, q: u64, seed: u64, cuda_stream: *mut c_void) -> i32;
    pub fn qf_version() -> *const c_char;
}
