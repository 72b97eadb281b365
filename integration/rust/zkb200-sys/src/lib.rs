//! zkb200-sys: raw bindings to libzkb200.so (GENERATED from include/zkb200.h by tools/gen_rust_ffi.py -- do not edit).
//! Conventions are those of risc0-sys: every operator returns NULL or a malloc'd message (`ffi_wrap`).
#![allow(non_camel_case_types)]
use std::ffi::{c_char, c_int, c_void, CStr};

#[repr(C)] pub struct ZkbCtx { _private: [u8; 0] }
#[repr(C)] pub struct ZkbProver { _private: [u8; 0] }
#[repr(C)] pub struct ZkbProgram { _private: [u8; 0] }
#[repr(C)] pub struct ZkbSession { _private: [u8; 0] }
pub type ZkbErr = *const c_char;

#[link(name = "zkb200")]
extern "C" {
    pub fn zkb_version() -> *const c_char;
    pub fn zkb_free_error(err: *const c_char);
    pub fn zkb_init(device: c_int, out: *mut *mut ZkbCtx) -> ZkbErr;
    pub fn zkb_init_on_stream(device: c_int, cuda_stream: *mut c_void, out: *mut *mut ZkbCtx) -> ZkbErr;
    pub fn zkb_destroy(ctx: *mut ZkbCtx) -> ZkbErr;
    pub fn zkb_sync(ctx: *mut ZkbCtx) -> ZkbErr;
    pub fn zkb_device_info(ctx: *mut ZkbCtx, sm_count: *mut c_int, cc_major: *mut c_int, cc_minor: *mut c_int, total_mem: *mut usize) -> ZkbErr;
    pub fn zkb_device_count(out: *mut c_int) -> ZkbErr;
    pub fn zkb_kernel_launches(ctx: *mut ZkbCtx, out: *mut u64) -> ZkbErr;
    pub fn zkb_timer_start(ctx: *mut ZkbCtx) -> ZkbErr;
    pub fn zkb_timer_stop(ctx: *mut ZkbCtx, ms: *mut f32) -> ZkbErr;
    pub fn zkb_alloc(ctx: *mut ZkbCtx, bytes: usize, d_out: *mut *mut c_void) -> ZkbErr;
    pub fn zkb_free(ctx: *mut ZkbCtx, d_ptr: *mut c_void) -> ZkbErr;
    pub fn zkb_host_alloc(ctx: *mut ZkbCtx, bytes: usize, h_out: *mut *mut c_void) -> ZkbErr;
    pub fn zkb_host_free(ctx: *mut ZkbCtx, h_ptr: *mut c_void) -> ZkbErr;
    pub fn zkb_memset0(ctx: *mut ZkbCtx, d_ptr: *mut c_void, bytes: usize) -> ZkbErr;
    pub fn zkb_fill_u32(ctx: *mut ZkbCtx, d_ptr: *mut c_void, n: usize, value: u32) -> ZkbErr;
    pub fn zkb_h2d(ctx: *mut ZkbCtx, d_dst: *mut c_void, h_src: *const c_void, bytes: usize) -> ZkbErr;
    pub fn zkb_d2h(ctx: *mut ZkbCtx, h_dst: *mut c_void, d_src: *const c_void, bytes: usize) -> ZkbErr;
    pub fn zkb_d2d(ctx: *mut ZkbCtx, d_dst: *mut c_void, d_src: *const c_void, bytes: usize) -> ZkbErr;
    pub fn zkb_batch_interpolate_ntt(ctx: *mut ZkbCtx, d_io: *mut c_void, count: usize, po2: c_int) -> ZkbErr;
    pub fn zkb_zk_shift(ctx: *mut ZkbCtx, d_io: *mut c_void, count: usize, po2: c_int) -> ZkbErr;
    pub fn zkb_batch_interpolate_ntt_zk_shift(ctx: *mut ZkbCtx, d_io: *mut c_void, count: usize, po2: c_int) -> ZkbErr;
    pub fn zkb_batch_expand(ctx: *mut ZkbCtx, d_out: *mut c_void, d_in: *const c_void, count: usize, in_po2: c_int, expand_bits: c_int) -> ZkbErr;
    pub fn zkb_batch_evaluate_ntt(ctx: *mut ZkbCtx, d_io: *mut c_void, count: usize, po2: c_int, expand_bits: c_int) -> ZkbErr;
    pub fn zkb_batch_expand_into_evaluate_ntt(ctx: *mut ZkbCtx, d_out: *mut c_void, d_in: *const c_void, count: usize, in_po2: c_int, expand_bits: c_int) -> ZkbErr;
    pub fn zkb_batch_bit_reverse(ctx: *mut ZkbCtx, d_io: *mut c_void, count: usize, po2: c_int) -> ZkbErr;
    pub fn zkb_poseidon2_hash_rows(ctx: *mut ZkbCtx, d_out_digests: *mut c_void, d_matrix: *const c_void, rows: usize, cols: usize) -> ZkbErr;
    pub fn zkb_poseidon2_hash_fold(ctx: *mut ZkbCtx, d_nodes: *mut c_void, input_size: usize, output_size: usize) -> ZkbErr;
    pub fn zkb_poseidon2_merkle_build(ctx: *mut ZkbCtx, d_nodes: *mut c_void, rows: usize) -> ZkbErr;
    pub fn zkb_batch_evaluate_any(ctx: *mut ZkbCtx, d_coeffs: *const c_void, poly_count: usize, po2: c_int, d_which: *const c_void, d_xs: *const c_void, d_out: *mut c_void, n_eval: usize) -> ZkbErr;
    pub fn zkb_mix_poly_coeffs(ctx: *mut ZkbCtx, d_out: *mut c_void, h_mix_start: *const u32, h_mix: *const u32, d_in: *const c_void, d_combos: *const c_void, input_size: usize, count: usize) -> ZkbErr;
    pub fn zkb_poly_divide(ctx: *mut ZkbCtx, d_poly: *mut c_void, n: usize, h_z: *const u32, d_rem: *mut c_void) -> ZkbErr;
    pub fn zkb_combos_divide(ctx: *mut ZkbCtx, d_combos: *mut c_void, n: usize, n_combos: usize, h_combo: *const u32, h_points: *const u32, n_div: usize, h_rem: *mut u32) -> ZkbErr;
    pub fn zkb_eltwise_sum_extelem(ctx: *mut ZkbCtx, d_out: *mut c_void, d_in: *const c_void, count: usize, to_add: usize) -> ZkbErr;
    pub fn zkb_fri_fold(ctx: *mut ZkbCtx, d_out: *mut c_void, d_in: *const c_void, h_mix: *const u32, out_count: usize) -> ZkbErr;
    pub fn zkb_eltwise_add_elem(ctx: *mut ZkbCtx, d_out: *mut c_void, d_a: *const c_void, d_b: *const c_void, n: usize) -> ZkbErr;
    pub fn zkb_eltwise_copy_elem(ctx: *mut ZkbCtx, d_out: *mut c_void, d_in: *const c_void, n: usize) -> ZkbErr;
    pub fn zkb_eltwise_zeroize_elem(ctx: *mut ZkbCtx, d_io: *mut c_void, n: usize) -> ZkbErr;
    pub fn zkb_gather_sample(ctx: *mut ZkbCtx, d_dst: *mut c_void, d_src: *const c_void, idx: usize, size: usize, stride: usize) -> ZkbErr;
    pub fn zkb_gather_rows(ctx: *mut ZkbCtx, d_dst: *mut c_void, d_src: *const c_void, src_len: usize, h_idx: *const u32, n_idx: usize, size: usize, stride: usize) -> ZkbErr;
    pub fn zkb_prefix_products(ctx: *mut ZkbCtx, d_io_fp4: *mut c_void, n: usize) -> ZkbErr;
    pub fn zkb_scatter(ctx: *mut ZkbCtx, d_into: *mut c_void, into_len: usize, h_index: *const u32, n_rows: usize, h_offsets: *const u32, h_values: *const u32) -> ZkbErr;
    pub fn zkb_eval_check(ctx: *mut ZkbCtx, d_check: *mut c_void, h_circuit: *const u32, circuit_words: usize, d_accum: *const c_void, d_code: *const c_void, d_data: *const c_void, h_mix_g: *const u32, h_out_g: *const u32, h_poly_mix: *const u32, po2: c_int) -> ZkbErr;
    pub fn zkb_eval_check_source(h_circuit: *const u32, circuit_words: usize, out: *mut c_char, cap: usize, needed: *mut usize) -> ZkbErr;
    pub fn zkb_eval_check_precompile(h_circuit: *const u32, circuit_words: usize) -> ZkbErr;
    pub fn zkb_accumulate(ctx: *mut ZkbCtx, h_circuit: *const u32, circuit_words: usize, d_accum: *mut c_void, d_code: *const c_void, d_data: *const c_void, h_mix: *const u32, h_io: *const u32, po2: c_int) -> ZkbErr;
    pub fn zkb_prover_new(ctx: *mut ZkbCtx, h_circuit: *const u32, circuit_words: usize, out: *mut *mut ZkbProver) -> ZkbErr;
    pub fn zkb_prover_free(p: *mut ZkbProver) -> ZkbErr;
    pub fn zkb_prover_segment_begin(p: *mut ZkbProver, po2: c_int, h_io: *const u32, code: *const c_void, data: *const c_void, traces_on_device: c_int, h_mix_out: *mut u32) -> ZkbErr;
    pub fn zkb_prover_segment_finish(p: *mut ZkbProver, accum: *const c_void, trace_on_device: c_int) -> ZkbErr;
    pub fn zkb_prover_seal_words(p: *mut ZkbProver, out: *mut usize) -> ZkbErr;
    pub fn zkb_prover_seal_copy(p: *mut ZkbProver, h_out: *mut u32) -> ZkbErr;
    pub fn zkb_prover_root_count(p: *mut ZkbProver, out: *mut usize) -> ZkbErr;
    pub fn zkb_prover_roots_copy(p: *mut ZkbProver, h_out: *mut u32) -> ZkbErr;
    pub fn zkb_prove_segment(p: *mut ZkbProver, po2: c_int, h_io: *const u32, code: *const c_void, data: *const c_void, accum: *const c_void, traces_on_device: c_int) -> ZkbErr;
    pub fn zkb_prover_stage_traces(p: *mut ZkbProver, po2: c_int, h_code: *const c_void, h_data: *const c_void, h_accum: *const c_void) -> ZkbErr;
    pub fn zkb_prove_staged(p: *mut ZkbProver, h_io: *const u32) -> ZkbErr;
    pub fn zkb_prover_stage_wait(p: *mut ZkbProver) -> ZkbErr;
    pub fn zkb_program_new(ctx: *mut ZkbCtx, h_circuit: *const u32, circuit_words: usize, out: *mut *mut ZkbProgram) -> ZkbErr;
    pub fn zkb_program_commit(prog: *mut ZkbProgram, po2: c_int, code: *const c_void, code_on_device: c_int, h_control_id: *mut u32) -> ZkbErr;
    pub fn zkb_program_control_ids(prog: *mut ZkbProgram, n: *mut usize, h_out: *mut u32) -> ZkbErr;
    pub fn zkb_program_free(prog: *mut ZkbProgram) -> ZkbErr;
    pub fn zkb_prover_set_program(p: *mut ZkbProver, prog: *mut ZkbProgram) -> ZkbErr;
    pub fn zkb_session_new(h_circuit: *const u32, circuit_words: usize, devices: *const c_int, n_devices: usize, inflight: c_int, out: *mut *mut ZkbSession) -> ZkbErr;
    pub fn zkb_session_commit(s: *mut ZkbSession, po2: c_int, h_code: *const c_void, h_control_id: *mut u32) -> ZkbErr;
    pub fn zkb_session_control_ids(s: *mut ZkbSession, n: *mut usize, h_out: *mut u32) -> ZkbErr;
    pub fn zkb_session_submit(s: *mut ZkbSession, po2: c_int, h_io: *const u32, h_data: *const c_void, h_accum: *const c_void, ticket: *mut u64) -> ZkbErr;
    pub fn zkb_session_wait(s: *mut ZkbSession, ticket: u64, h_seal: *mut u32, words: *mut usize) -> ZkbErr;
    pub fn zkb_session_free(s: *mut ZkbSession) -> ZkbErr;
    pub fn zkb_verify_segment(h_circuit: *const u32, circuit_words: usize, h_seal: *const u32, seal_words: usize, h_control_ids: *const u32, n_control_ids: usize, h_out_po2_code_root: *mut u32) -> ZkbErr;
    pub fn zkb_poseidon254_hash_rows(ctx: *mut ZkbCtx, d_out_digests: *mut c_void, d_matrix: *const c_void, rows: usize, cols: usize) -> ZkbErr;
    pub fn zkb_poseidon254_hash_fold(ctx: *mut ZkbCtx, d_nodes: *mut c_void, input_size: usize, output_size: usize) -> ZkbErr;
    pub fn zkb_poseidon254_merkle_build(ctx: *mut ZkbCtx, d_nodes: *mut c_void, rows: usize) -> ZkbErr;
    pub fn zkb_poseidon254_permute_host(h_in: *const u32, h_out: *mut u32) -> ZkbErr;
}

/// NULL = Ok; otherwise copy the message, free it with zkb_free_error and return it as an error (risc0-sys `ffi_wrap`).
pub fn ffi_wrap<F: FnOnce() -> ZkbErr>(f: F) -> Result<(), String> {
    let e = f();
    if e.is_null() { return Ok(()); }
    let msg = unsafe { CStr::from_ptr(e) }.to_string_lossy().into_owned();
    unsafe { zkb_free_error(e) };
    Err(msg)
}
