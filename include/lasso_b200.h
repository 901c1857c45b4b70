/* lasso_b200 — C ABI of the B200-native Lasso prover hot path.
 *
 * This is the drop-in boundary for a16z/Lasso's
 *   DensifiedRepresentation::from_lookup_indices -> commit -> SparsePolynomialEvaluationProof::prove
 * path (SURVEY.md §8b).  The reference has no FFI of its own (it is three Rust generics); each entry
 * point below names the reference item it replaces (file:line relative to the reference's src/),
 * which is where a Rust maintainer would bind it (see INTEGRATION.md for the extern "C" shim).
 *
 * Conventions
 *  - field elements (curve25519 Fr) are 4 x uint64_t little-endian limbs in ark-ff Montgomery form
 *    (a * 2^256 mod l): a Rust `&[Fr]` can be passed as `*const u64` without conversion;
 *  - affine points are (x, y) = 2 x 4 x uint64_t Fq Montgomery limbs (ark_ec TE `Affine`, 64 B);
 *    extended points are (x, y, t, z) = 4 x 4 x uint64_t (ark_ec TE `Projective`, 128 B);
 *  - every call is blocking; buffers are caller-owned HOST memory unless a name says otherwise;
 *  - return value 0 = ok; > 0 = the reference's panic / Err condition; < 0 = CUDA / internal error
 *    (lasso_last_error() gives the text).  There is no CPU fallback: without a CUDA device
 *    lasso_ctx_create fails and nothing else can be called.
 */
#ifndef LASSO_B200_H
#define LASSO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct lasso_ctx lasso_ctx;
typedef struct lasso_gens lasso_gens;   /* SparsePolyCommitmentGens<G>        lasso/surge.rs:25-58  */
typedef struct lasso_dense lasso_dense; /* DensifiedRepresentation<F, C>      lasso/densified.rs:8-18 */

/* SubtableStrategy impls (subtables/{and,or,xor,lt,range_check}.rs) */
enum { LASSO_AND = 0, LASSO_OR = 1, LASSO_XOR = 2, LASSO_LT = 3, LASSO_RANGE_CHECK = 4 };

/* error codes > 0 mirror the reference's panics */
enum {
  LASSO_OK = 0,
  LASSO_ERR_LENGTH = 1,      /* assert_eq!(r.len(), log2(s)) surge.rs:131; msm Err(min_len) msm/mod.rs:36-40 */
  LASSO_ERR_NOT_POW2 = 2,    /* DensePolynomial::new on a non power of two  poly/dense_mlpoly.rs:63-66 */
  LASSO_ERR_INDEX_RANGE = 3, /* debug_assert!(memory_address < m)           lasso/densified.rs:46 */
  LASSO_ERR_STRATEGY = 4,    /* unknown / unsupported strategy parameters */
  LASSO_ERR_GENS = 5,        /* generator set too small for the polynomial  poly/commitments.rs:85 */
  LASSO_ERR_MULTISET = 6     /* assert_eq!(hash_init*hash_write, hash_read*hash_final) memory_checking.rs:689 */
};

const char* lasso_last_error(void);

/* One context per GPU: owns the device, stream, memory pool and scratch. */
int lasso_ctx_create(lasso_ctx** out, int device_id);
void lasso_ctx_destroy(lasso_ctx* ctx);

/* One proof sharded over `world` ranks of ONE node (one process per GPU, world a power of two <= 8; several ranks
 * may also share a GPU): rank 0 obtains an id with lasso_comm_unique_id, every rank receives it out of band (e.g.
 * torch.distributed broadcast) and calls lasso_ctx_init_comm before any other call.  Afterwards lasso_densify /
 * lasso_commit / lasso_prove are collective: every rank passes the SAME arguments, holds the low-index-bit shard
 * of every polynomial, and receives the same (bit-identical to single-GPU) commitment and proof bytes.
 * Exchanges (DESIGN.md section 6): per sumcheck round every GPU stores its three partial sums into the shared
 * pinned host segment of every process (no collective, no extra launch); the few bulk hand-overs (partial points
 * of a row-MSM, heads of the polynomials, the LZ vector of an opening) are all-gathers written as one kernel of
 * peer-memory stores over NVLink (CUDA IPC), or ncclAllGather under LASSO_B200_XCHG=nccl. */
int lasso_comm_unique_id(uint8_t out[128]);
int lasso_ctx_init_comm(lasso_ctx*, const uint8_t id[128], int rank, int world);
/* Optional host-thread placement for one process per GPU on a multi-socket node (sysfs; returns the NUMA node of the
 * context's GPU, or -1 if the topology is not exposed): the CALLING thread — the one that will call lasso_prove and
 * spin on the round messages — is pinned to a dedicated physical core of that node (a different one for every GPU
 * of the node), the library's helper threads (staging of the index matrix) get the rest of the node.  Call it from
 * the proving thread after the process has created its other threads (they keep their affinity). */
int lasso_ctx_bind_host_threads(lasso_ctx*);

/* ---------------------------------------------------------------- per-loop entry points (host buffers) */

/* DensePolynomial::bound_poly_var_top  poly/dense_mlpoly.rs:209-216.  Z has `len` elements; the first
 * len/2 are overwritten with the bound polynomial. */
int lasso_bind_top(lasso_ctx*, uint64_t* Z, size_t len, const uint64_t r[4]);
/* DensePolynomial::bound_poly_var_bot  poly/dense_mlpoly.rs:218-225 */
int lasso_bind_bot(lasso_ctx*, uint64_t* Z, size_t len, const uint64_t r[4]);
/* EqPolynomial::evals  poly/eq_poly.rs:21-38.  out has 2^ell elements; r[0] binds the MSB. */
int lasso_eq_evals(lasso_ctx*, const uint64_t* r, int ell, uint64_t* out);
/* One round of SumcheckInstanceProof::prove_arbitrary's evaluation loop  subprotocols/sumcheck.rs:179-237
 * with comb_func = S::combine_lookups_eq.  polys = (NUM_MEMORIES+1) arrays of `len` elements, the last
 * one the eq polynomial.  evals_out receives sumcheck_poly_degree()+1 elements (t = 0..deg). */
int lasso_sumcheck_round_arbitrary(lasso_ctx*, int strategy, int C, int log_M, int log_R,
                                   const uint64_t* const* polys, size_t len, uint64_t* evals_out);
/* The step between two rounds of prove_arbitrary as the prover runs it: bind every polynomial's top variable to r
 * (subprotocols/sumcheck.rs:247-253, in place: polys[k][0 .. len/2) are overwritten), then evaluate the next
 * round over the bound polynomials (sumcheck.rs:179-237).  One fused pass for the strategies with a linear g.
 * len >= 4. */
int lasso_sumcheck_bind_round_arbitrary(lasso_ctx*, int strategy, int C, int log_M, int log_R, uint64_t* const* polys,
                                        size_t len, const uint64_t r[4], uint64_t* evals_out);
/* One round of prove_cubic_batched's evaluation loop  subprotocols/sumcheck.rs:49-93:
 * e0e2e3_out[3k..3k+3) = sum_i A_k B_k Ceq at t = 0, 2, 3. */
int lasso_sumcheck_round_cubic(lasso_ctx*, int n_circuits, const uint64_t* const* A, const uint64_t* const* B,
                               const uint64_t* Ceq, size_t len, uint64_t* e0e2e3_out);
/* SubtableStrategy::materialize_subtables  subtables/{and.rs:16-28,or.rs,xor.rs:16-27,lt.rs:16-30,
 * range_check.rs:15-34}.  tables_out[k] has M = 2^log_M elements, k < NUM_SUBTABLES. */
int lasso_materialize_subtables(lasso_ctx*, int strategy, int C, int log_M, int log_R, uint64_t* const* tables_out);
/* SubtableStrategy::to_lookup_polys  subtables/mod.rs:78-92.  nz[d] = lookup indices of dimension d
 * (s entries, `usize` = u64); E_out[k] receives s elements, k < NUM_MEMORIES. */
int lasso_gather_lookup_polys(lasso_ctx*, int strategy, int C, int log_M, int log_R, const uint64_t* const* nz,
                              size_t s, uint64_t* const* E_out);
/* VariableBaseMSM::msm  msm/mod.rs:36-40 (bases: n affine points, scalars: n Fr) -> one extended point,
 * normalised (z = 1).  Same group element as the reference's msm_bigint_wnaf.  After lasso_ctx_init_comm this
 * (and lasso_commit_rows) is collective: each rank passes ITS SHARD of the terms (any split), partial points are
 * all-gathered over NCCL and added, every rank receives the full sum. */
int lasso_msm(lasso_ctx*, const uint64_t* bases_affine, const uint64_t* scalars, size_t n, uint64_t out_xytz[16]);
/* BASELINE config 5 — the same VariableBaseMSM::msm on DEVICE-RESIDENT inputs, as a reusable job: `n` terms, term i
 * uses base i % n_pool (n_pool == n: one base per term; smaller: a pool of distinct points tiled, for benchmarks).
 * lasso_msm_job_run runs the whole MSM (scalars -> canonical integers, bases -> internal form, Pippenger with the
 * reference's window rule, msm/mod.rs:91-164) `iters` times between two CUDA events on the context's stream and
 * returns the average ms and the normalised point; info (may be null) = {window bits c, windows, widest scalar bits,
 * unit size, L, T2, world, 0}.  On a sharded context every rank passes ITS terms and the call is collective.
 * lasso_msm_job_naive evaluates the same sum by per-term double-and-add + a tree sum (an independent cross-check
 * for sizes the CPU oracle cannot reach). */
typedef struct lasso_msm_job lasso_msm_job;
/* The schedule the large MSM would use for n terms whose widest scalar has max_bits bits (no GPU needed): out = {window
 * bits c (the reference's rule, msm/mod.rs:112-116, capped at 17), windows, scalar bits, buckets per window 2^(c-1), unit
 * size, reduction levels, group size of level 0.., zero padded}. */
int lasso_msm_plan_info(size_t n, unsigned max_bits, int out[16]);
int lasso_msm_job_create(lasso_ctx*, const uint64_t* bases_affine, size_t n_pool, const uint64_t* scalars, size_t n,
                         lasso_msm_job** out);
int lasso_msm_job_run(lasso_ctx*, lasso_msm_job*, int iters, double* avg_ms, uint64_t out_xytz[16], int info[8]);
int lasso_msm_job_naive(lasso_ctx*, lasso_msm_job*, uint64_t out_xytz[16]);
void lasso_msm_job_destroy(lasso_msm_job*);
/* DensePolynomial::commit_inner  poly/dense_mlpoly.rs:109-128 (+ Commitments::batch_commit
 * poly/commitments.rs:84-93 with blind = 0): Z viewed as L_size rows of R_size; gens_affine holds the
 * R_size generators followed by h.  out_points = L_size extended points (z = 1). */
int lasso_commit_rows(lasso_ctx*, const uint64_t* gens_affine, const uint64_t* Z, size_t L_size, size_t R_size,
                      uint64_t* out_points);

/* ---------------------------------------------------------------- the whole path, device-resident */

/* Number of generator-stream points SparsePolyCommitmentGens::new(label, c, s, num_memories, log_m)
 * needs (the widest PolyCommitmentGens: n + 2).  lasso/surge.rs:32-58, subprotocols/dot_product.rs:146-149 */
size_t lasso_gens_points_needed(size_t c, size_t s, size_t num_memories, size_t log_m);
/* MultiCommitGens::new's sampling (poly/commitments.rs:22-44): Shake256(label || compressed generator)
 * -> ChaCha20Rng -> G::rand, `count` affine points.  Deterministic; see DESIGN.md on what is unpinned. */
int lasso_sample_generators(const char* label, size_t count, uint64_t* out_affine);
/* SparsePolyCommitmentGens from an explicit generator stream (the parity contract passes generators in):
 * stream[0..n) = G, stream[n] = gens_1.G[0], stream[n+1] = h for each of the three PolyCommitmentGens.
 * Also expands the stream into the fixed-base window table and — on a single-GPU context — the digit-multiples
 * tables of the opening / commitment generators (DESIGN.md section 2: ~14 GB of HBM at 2^20 lookups;
 * LASSO_B200_NO_MULTIPLES=1 disables them, LASSO_B200_TABLE_GB caps the 16-bit one).  Outputs do not depend on it. */
int lasso_gens_create(lasso_ctx*, const uint64_t* stream_affine, size_t n_points, size_t c, size_t s,
                      size_t num_memories, size_t log_m, lasso_gens** out);
void lasso_gens_destroy(lasso_gens*);

/* DensifiedRepresentation::from_lookup_indices  lasso/densified.rs:21-75.
 * indices: n_lookups x C row-major `usize` (the reference's &Vec<[usize; C]>). */
int lasso_densify(lasso_ctx*, const uint64_t* indices, size_t n_lookups, size_t C, size_t log_m, lasso_dense** out);
/* Element types of lasso_densify_device's index matrix. */
enum { LASSO_IDX_U64 = 0, LASSO_IDX_I64 = 1, LASSO_IDX_U32 = 2, LASSO_IDX_I32 = 3 };
/* DensifiedRepresentation::from_lookup_indices (lasso/densified.rs:21-75) on DEVICE-RESIDENT indices: the same result as
 * lasso_densify, read in place from memory of the context's device (cudaMalloc'd or managed; e.g. a CUDA tensor).
 * Element (k, d) of the n_lookups x C matrix is indices[k * row_stride + d * col_stride], strides in elements and >= 0
 * (row-major: C, 1; column-major: 1, n_lookups; one column broadcast to all C dimensions: 1, 0), of type dtype
 * (LASSO_IDX_*).  A negative index or one >= 2^log_m returns LASSO_ERR_INDEX_RANGE; bad shapes, strides or dtype
 * LASSO_ERR_STRATEGY; a pointer that is not memory of the context's device < 0, before anything is allocated or
 * launched.  The extent of the buffer is not checked: it must hold every element the strides address.
 * Ordering: the call first waits (on the device) for the work already queued on cuda_stream (a cudaStream_t of the
 * context's device; NULL = the legacy default stream), so a producer may still be writing the matrix when it is called.
 * Lifetime: on return the library no longer reads the buffer; the caller may overwrite or free it at once.
 * Sharded (after lasso_ctx_init_comm): collective, every rank passes a matrix with the same contents on its own device,
 * and every rank reports the same result. */
int lasso_densify_device(lasso_ctx*, const void* indices, int dtype, size_t n_lookups, size_t C, int64_t row_stride,
                         int64_t col_stride, size_t log_m, void* cuda_stream, lasso_dense** out);
void lasso_dense_destroy(lasso_dense*);
size_t lasso_dense_s(const lasso_dense*);
/* copies of the public fields (densified.rs:8-18) back to the host, for inspection / tests:
 * which = 0 dim_usize (C*s u64), 1 dim (C*s Fr), 2 read (C*s Fr), 3 final (C*m Fr),
 *         4 combined_l_variate_polys (Fr), 5 combined_log_m_variate_polys (Fr).  Returns element count. */
size_t lasso_dense_read(lasso_ctx*, const lasso_dense*, int which, uint64_t* out, size_t cap_elems);

/* DensifiedRepresentation::commit  lasso/densified.rs:77-96 -> SparsePolynomialCommitment serialised with
 * ark-serialize (compressed): Vec<G> l_variate, Vec<G> log_m_variate, s, log_m, m (surge.rs:61-68). */
int lasso_commit(lasso_ctx*, const lasso_dense*, const lasso_gens*, uint8_t* out, size_t cap, size_t* out_len);

/* SparsePolynomialEvaluationProof::<G, C, M, S>::prove  lasso/surge.rs:118-211.
 * r: log2(s) Fr elements.  transcript_label: Transcript::new(label) (b"example" in bench.rs:59);
 * tape_label / tape_seed: RandomTape::new(b"proof") seeded with an explicit scalar (the reference draws it
 * from ark_std::test_rng()).  proof_out receives the ark-serialize (compressed) bytes of the proof struct.
 * challenges_out (optional) receives every Fiat-Shamir challenge in order (4 limbs each). */
int lasso_prove(lasso_ctx*, int strategy, int log_R, lasso_dense*, const uint64_t* r, size_t r_len,
                const lasso_gens*, const char* transcript_label, const char* tape_label, const uint64_t tape_seed[4],
                uint8_t* proof_out, size_t proof_cap, size_t* proof_len, uint64_t* challenges_out,
                size_t challenges_cap, size_t* n_challenges);

/* Host-resident benchmark helper: number of kernels launched by this context so far, and the wall time
 * (ms) of the last densify / commit / prove calls. */
unsigned long long lasso_launch_count(const lasso_ctx*);
void lasso_last_timings(const lasso_ctx*, double out_ms[3]);
/* With LASSO_B200_SPANS=1 in the environment the prover synchronises around named spans (the analogue of the
 * reference's tracing spans, e.g. "Sumcheck.prove", "Subtables.commit"); this drains them as "name=ms;..." */
size_t lasso_spans(const lasso_ctx*, char* buf, size_t cap);

/* Device-resident bind benchmark hook (bench.py roofline leg): allocates npolys x len random elements on the
 * device once, then runs `iters` top-binds over them on the context stream and returns the average kernel
 * duration in ms measured with CUDA events on that stream. */
int lasso_bench_bind(lasso_ctx*, size_t len, int npolys, int iters, double* avg_ms);

#ifdef __cplusplus
}
#endif
#endif
