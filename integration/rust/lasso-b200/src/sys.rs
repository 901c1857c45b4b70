//! Raw declarations of include/lasso_b200.h (one per C entry point; the header cites the reference item each replaces).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct lasso_ctx {
    _p: [u8; 0],
}
#[repr(C)]
pub struct lasso_gens {
    _p: [u8; 0],
}
#[repr(C)]
pub struct lasso_dense {
    _p: [u8; 0],
}
#[repr(C)]
pub struct lasso_msm_job {
    _p: [u8; 0],
}

extern "C" {
    pub fn lasso_last_error() -> *const c_char;
    pub fn lasso_ctx_create(out: *mut *mut lasso_ctx, device_id: c_int) -> c_int;
    pub fn lasso_ctx_destroy(ctx: *mut lasso_ctx);
    pub fn lasso_comm_unique_id(out: *mut u8) -> c_int;
    pub fn lasso_ctx_init_comm(ctx: *mut lasso_ctx, id: *const u8, rank: c_int, world: c_int) -> c_int;
    pub fn lasso_ctx_bind_host_threads(ctx: *mut lasso_ctx) -> c_int;
    // per-loop entry points (host buffers)
    pub fn lasso_bind_top(ctx: *mut lasso_ctx, z: *mut u64, len: usize, r: *const u64) -> c_int;
    pub fn lasso_bind_bot(ctx: *mut lasso_ctx, z: *mut u64, len: usize, r: *const u64) -> c_int;
    pub fn lasso_eq_evals(ctx: *mut lasso_ctx, r: *const u64, ell: c_int, out: *mut u64) -> c_int;
    pub fn lasso_sumcheck_round_arbitrary(ctx: *mut lasso_ctx, strategy: c_int, c: c_int, log_m: c_int, log_r: c_int,
                                          polys: *const *const u64, len: usize, evals_out: *mut u64) -> c_int;
    pub fn lasso_sumcheck_bind_round_arbitrary(ctx: *mut lasso_ctx, strategy: c_int, c: c_int, log_m: c_int, log_r: c_int,
                                               polys: *const *mut u64, len: usize, r: *const u64, evals_out: *mut u64) -> c_int;
    pub fn lasso_sumcheck_round_cubic(ctx: *mut lasso_ctx, n_circuits: c_int, a: *const *const u64, b: *const *const u64,
                                      ceq: *const u64, len: usize, e0e2e3_out: *mut u64) -> c_int;
    pub fn lasso_materialize_subtables(ctx: *mut lasso_ctx, strategy: c_int, c: c_int, log_m: c_int, log_r: c_int,
                                       tables_out: *const *mut u64) -> c_int;
    pub fn lasso_gather_lookup_polys(ctx: *mut lasso_ctx, strategy: c_int, c: c_int, log_m: c_int, log_r: c_int,
                                     nz: *const *const u64, s: usize, e_out: *const *mut u64) -> c_int;
    pub fn lasso_msm(ctx: *mut lasso_ctx, bases: *const u64, scalars: *const u64, n: usize, out_xytz: *mut u64) -> c_int;
    pub fn lasso_commit_rows(ctx: *mut lasso_ctx, gens: *const u64, z: *const u64, l_size: usize, r_size: usize,
                             out_points: *mut u64) -> c_int;
    pub fn lasso_msm_plan_info(n: usize, max_bits: u32, out: *mut c_int) -> c_int;
    pub fn lasso_msm_job_create(ctx: *mut lasso_ctx, bases: *const u64, n_pool: usize, scalars: *const u64, n: usize,
                                out: *mut *mut lasso_msm_job) -> c_int;
    pub fn lasso_msm_job_run(ctx: *mut lasso_ctx, job: *mut lasso_msm_job, iters: c_int, avg_ms: *mut f64, out_xytz: *mut u64,
                             info: *mut c_int) -> c_int;
    pub fn lasso_msm_job_naive(ctx: *mut lasso_ctx, job: *mut lasso_msm_job, out_xytz: *mut u64) -> c_int;
    pub fn lasso_msm_job_destroy(job: *mut lasso_msm_job);
    // the whole path, device resident
    pub fn lasso_gens_points_needed(c: usize, s: usize, num_memories: usize, log_m: usize) -> usize;
    pub fn lasso_sample_generators(label: *const c_char, count: usize, out_affine: *mut u64) -> c_int;
    pub fn lasso_gens_create(ctx: *mut lasso_ctx, stream: *const u64, n_points: usize, c: usize, s: usize, num_memories: usize,
                             log_m: usize, out: *mut *mut lasso_gens) -> c_int;
    pub fn lasso_gens_destroy(g: *mut lasso_gens);
    pub fn lasso_densify(ctx: *mut lasso_ctx, indices: *const u64, n_lookups: usize, c: usize, log_m: usize,
                         out: *mut *mut lasso_dense) -> c_int;
    // indices: device memory of the context's device; dtype: LASSO_IDX_{U64 = 0, I64 = 1, U32 = 2, I32 = 3};
    // cuda_stream: a cudaStream_t (null = legacy default stream)
    pub fn lasso_densify_device(ctx: *mut lasso_ctx, indices: *const c_void, dtype: c_int, n_lookups: usize, c: usize,
                                row_stride: i64, col_stride: i64, log_m: usize, cuda_stream: *mut c_void,
                                out: *mut *mut lasso_dense) -> c_int;
    pub fn lasso_dense_destroy(d: *mut lasso_dense);
    pub fn lasso_dense_s(d: *const lasso_dense) -> usize;
    pub fn lasso_dense_read(ctx: *mut lasso_ctx, d: *const lasso_dense, which: c_int, out: *mut u64, cap_elems: usize) -> usize;
    pub fn lasso_commit(ctx: *mut lasso_ctx, d: *const lasso_dense, g: *const lasso_gens, out: *mut u8, cap: usize,
                        out_len: *mut usize) -> c_int;
    pub fn lasso_prove(ctx: *mut lasso_ctx, strategy: c_int, log_r: c_int, d: *mut lasso_dense, r: *const u64, r_len: usize,
                       g: *const lasso_gens, transcript_label: *const c_char, tape_label: *const c_char, tape_seed: *const u64,
                       proof_out: *mut u8, proof_cap: usize, proof_len: *mut usize, challenges_out: *mut u64,
                       challenges_cap: usize, n_challenges: *mut usize) -> c_int;
    pub fn lasso_launch_count(ctx: *const lasso_ctx) -> u64;
    pub fn lasso_last_timings(ctx: *const lasso_ctx, out_ms: *mut f64);
}
