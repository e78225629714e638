//! `extern "C"` declarations mirroring include/zkb200.h one to one.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_void};

#[repr(C)]
pub struct zkb_ctx {
    _private: [u8; 0],
}

#[repr(C)]
pub struct zkb_air_desc {
    pub air_id: u32,
    pub trace_width: u32,
    pub trace_len: u64,
    pub num_queries: u32,
    pub blowup: u32,
    pub grinding_bits: u32,
    pub field_extension: u32,
    pub folding: u32,
    pub rem_max_degree: u32,
    pub batching_constraints: u32,
    pub batching_deep: u32,
    pub pub_elems: *const u8,
    pub n_pub_elems: u64,
    pub assert_cols: *const u32,
    pub assert_steps: *const u64,
    pub assert_values: *const u8,
    pub n_assertions: u64,
    pub params: *const u8,
    pub n_params: u64,
}

#[repr(C)]
pub struct zkb_transcript {
    pub trace_root: [u8; 32],
    pub constraint_root: [u8; 32],
    pub remainder_commitment: [u8; 32],
    pub constraint_alpha: [u8; 16],
    pub z: [u8; 16],
    pub deep_alpha: [u8; 16],
    pub n_fri_layers: u32,
    pub n_positions: u32,
    pub fri_roots: [[u8; 32]; 16],
    pub fri_alphas: [[u8; 16]; 16],
    pub pow_nonce: u64,
    pub positions: [u32; 256],
    pub comp_degree_ok: i32,
    pub _pad: i32,
}

pub const ZKB_AIR_ID_TRAINING: u32 = 1;
pub const ZKB_AIR_ID_AGGREGATION: u32 = 2;
pub const ZKB_AIR_ID_MIMC: u32 = 3;

/// zkb_verdict: one value per check of winter-verifier's `verify`, in the order it runs them
pub const ZKB_VERIFY_OK: i32 = 0;
pub const ZKB_VERIFY_MALFORMED: i32 = 1;
pub const ZKB_VERIFY_TRACE_INFO: i32 = 2;
pub const ZKB_VERIFY_OPTIONS: i32 = 3;
pub const ZKB_VERIFY_COMMITMENTS: i32 = 4;
pub const ZKB_VERIFY_OOD_FRAME: i32 = 5;
pub const ZKB_VERIFY_OOD_CONSISTENCY: i32 = 6;
pub const ZKB_VERIFY_POW: i32 = 7;
pub const ZKB_VERIFY_UNIQUE_QUERIES: i32 = 8;
pub const ZKB_VERIFY_TRACE_VALUES: i32 = 9;
pub const ZKB_VERIFY_TRACE_MERKLE: i32 = 10;
pub const ZKB_VERIFY_CONSTRAINT_VALUES: i32 = 11;
pub const ZKB_VERIFY_CONSTRAINT_MERKLE: i32 = 12;
pub const ZKB_VERIFY_FRI_VALUES: i32 = 13;
pub const ZKB_VERIFY_FRI_MERKLE: i32 = 14;
pub const ZKB_VERIFY_FRI_FOLDING: i32 = 15;
pub const ZKB_VERIFY_FRI_TRUNCATION: i32 = 16;
pub const ZKB_VERIFY_REMAINDER_DEGREE: i32 = 17;
pub const ZKB_VERIFY_REMAINDER_COMMITMENT: i32 = 18;
pub const ZKB_VERIFY_REMAINDER_FOLDING: i32 = 19;

extern "C" {
    pub fn zkb_ctx_create(device: i32, stream: *mut c_void, out: *mut *mut zkb_ctx) -> i32;
    pub fn zkb_ctx_create_lane(device: i32, out: *mut *mut zkb_ctx) -> i32;
    pub fn zkb_ctx_destroy(ctx: *mut zkb_ctx);
    pub fn zkb_last_error(ctx: *const zkb_ctx) -> *const c_char;
    pub fn zkb_free(p: *mut c_void);

    pub fn zkb_prove(ctx: *mut zkb_ctx, air: *const zkb_air_desc, cols: *const *const u8, force_nonce: u64,
                     proof_out: *mut *mut u8, proof_len: *mut u64, transcript: *mut zkb_transcript) -> i32;

    pub fn zkb_prove_device(ctx: *mut zkb_ctx, air: *const zkb_air_desc, d_trace_colmajor: *const c_void, force_nonce: u64,
                            proof_out: *mut *mut u8, proof_len: *mut u64, transcript: *mut zkb_transcript) -> i32;
    pub fn zkb_prove_batch(lanes: *const *mut zkb_ctx, n_lanes: u32, airs: *const *const zkb_air_desc, cols: *const *const *const u8,
                           count: u32, proofs_out: *mut *mut u8, lens_out: *mut u64) -> i32;
    /// winterfell::verify for `count` proofs; verdicts_out[i] = ZKB_VERIFY_OK (0) or the first zkb_verdict proof i fails
    pub fn zkb_verify_batch(ctx: *mut zkb_ctx, airs: *const *const zkb_air_desc, proofs: *const *const u8, lens: *const u64, count: u32,
                            verdicts_out: *mut i32, transcripts_out: *mut zkb_transcript) -> i32;
    /// key32: 32 bytes of ChaCha20 key for the blinding masks, or null = OS entropy (what rand::thread_rng() does)
    pub fn zkb_training_trace_device(ctx: *mut zkb_ctx, raw_rows: *const u8, n_raw: u32, half: u32, n: u64, key32: *const u8,
                                     d_out: *mut *mut c_void, first_row_out: *mut u8, last_row_out: *mut u8) -> i32;

    pub fn zkb_begin(ctx: *mut zkb_ctx, air: *const zkb_air_desc) -> i32;
    pub fn zkb_trace_commit(ctx: *mut zkb_ctx, cols: *const *const u8, root_out: *mut u8) -> i32;
    pub fn zkb_trace_read_frame(ctx: *mut zkb_ctx, lde_step: u64, current_out: *mut u8, next_out: *mut u8) -> i32;
    pub fn zkb_trace_read_frames(ctx: *mut zkb_ctx, lde_steps: *const u64, count: u32, current_out: *mut u8, next_out: *mut u8) -> i32;
    pub fn zkb_trace_polys_read(ctx: *mut zkb_ctx, out: *mut u8) -> i32;
    pub fn zkb_constraints_eval(ctx: *mut zkb_ctx, alpha: *const u8, evals_out: *mut u8) -> i32;
    pub fn zkb_constraints_commit(ctx: *mut zkb_ctx, root_out: *mut u8) -> i32;
    pub fn zkb_ood_eval(ctx: *mut zkb_ctx, z: *const u8, cur_out: *mut u8, next_out: *mut u8, h_out: *mut u8) -> i32;
    pub fn zkb_deep_compose(ctx: *mut zkb_ctx, deep_alpha: *const u8) -> i32;
    pub fn zkb_fri_num_layers(ctx: *mut zkb_ctx, out: *mut u32) -> i32;
    pub fn zkb_fri_commit_layer(ctx: *mut zkb_ctx, root_out: *mut u8) -> i32;
    pub fn zkb_fri_fold(ctx: *mut zkb_ctx, alpha: *const u8) -> i32;
    pub fn zkb_fri_remainder(ctx: *mut zkb_ctx, coeffs_out: *mut u8, n_coeffs_out: *mut u64, commitment_out: *mut u8) -> i32;
    pub fn zkb_grind(ctx: *mut zkb_ctx, seed: *const u8, bits: u32, nonce_out: *mut u64) -> i32;
    pub fn zkb_query(ctx: *mut zkb_ctx, which: u32, positions: *const u32, n_pos: u32, rows_out: *mut u8,
                     proof_out: *mut *mut u8, proof_len: *mut u64) -> i32;
}
