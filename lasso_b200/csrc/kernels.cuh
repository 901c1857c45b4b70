// lasso_b200 — launcher interface between the host prover / C-ABI and the CUDA kernels.
// All pointers are device pointers unless named h_*.  Every launcher is asynchronous on
// the given stream.
#pragma once
#include "common.cuh"

namespace lb {

enum StrategyKind { STRAT_AND = 0, STRAT_OR = 1, STRAT_XOR = 2, STRAT_LT = 3, STRAT_RANGE = 4 };

// Runtime stand-in for the reference's `impl SubtableStrategy<F, C, M>` const generics
// (src/subtables/mod.rs:31-93).
struct Strategy {
  int kind, C, log_m, log_r;
  int M() const { return 1 << log_m; }
  int num_subtables() const { return kind == STRAT_LT ? 2 : (kind == STRAT_RANGE ? 3 : 1); }
  int num_memories() const { return kind == STRAT_LT ? 2 * C : C; }
  int g_poly_degree() const { return kind == STRAT_LT ? C : 1; }
  int sumcheck_poly_degree() const { return g_poly_degree() + 1; }
  // src/subtables/mod.rs:64-74, range_check.rs:62-73
  int memory_to_subtable_index(int i) const {
    if (kind == STRAT_RANGE) {
      if (i * log_m > log_r) return 2;
      return ((i + 1) * log_m > log_r) ? 1 : 0;
    }
    return i % num_subtables();
  }
  int memory_to_dimension_index(int i) const { return kind == STRAT_RANGE ? i : i / num_subtables(); }
  bool valid() const {
    if (!(kind >= 0 && kind <= 4 && C >= 1 && C <= 16 && log_m >= 2 && log_m <= 24 && (log_m % 2 == 0 || kind == STRAT_RANGE)))
      return false;
    // combine_lookups weights are F::from(1u64 << (i * inc)) (and.rs:45-53, range_check.rs:78-86): the shift must
    // stay below 64 (the debug-build reference panics on overflow); RangeCheck<LOG_R> needs LOG_R >= 0
    if (kind != STRAT_LT && (num_memories() - 1) * (kind == STRAT_RANGE ? log_m : log_m / 2) >= 64) return false;
    if (kind == STRAT_RANGE && log_r < 0) return false;
    return true;
  }
};

struct FrVec {  // small vector passed by value as a kernel parameter (challenge points, weights)
  fr_t v[32];
};

// ---- K1: bind (dense_mlpoly.rs:209-225) ----
// Z_k[i] <- Z_k[i] + r (Z_k[i+half] - Z_k[i]) for k < npolys, Z_k = base + k*stride, i < half
void launch_bind_top(fr_t* base, size_t stride, int npolys, size_t half, const fr_t& r, cudaStream_t st);
// same over an array of independent device pointers (grand-product circuits)
void launch_bind_top_ptrs(fr_t* const* d_ptrs, int npolys, size_t half, const fr_t& r, cudaStream_t st);
// out[i] <- Z[2i] + r (Z[2i+1] - Z[2i]), out-of-place
void launch_bind_bot(const fr_t* Z, fr_t* out, size_t half, const fr_t& r, cudaStream_t st);

// ---- K4: eq evals (eq_poly.rs:21-38); scratch needs 2 * 4096 elements when ell > 12 ----
void launch_eq_evals(const FrVec& r, int ell, fr_t* out, fr_t* scratch, cudaStream_t st);

// ---- K2: primary sumcheck round evaluation (sumcheck.rs:179-237) ----
// polys = (alpha+1) arrays of length 2*half at base + k*stride (the last one is eq).
// One launch: the last CTA reduces the block partials and publishes the deg+1 results (see Finalize).
void launch_sumcheck_eval_arbitrary(const Strategy& S, const fr_t* base, size_t stride, size_t half, const Finalize& fin,
                                    cudaStream_t st);
// The previous round's bind (with r) fused with this round's evaluation: base holds polynomials of length 4q, bound
// in place to 2q.  Returns false (nothing launched) when the strategy has no fused kernel or q < min_q (0: the
// default threshold below which a round is latency-bound and two short launches are quicker).
bool launch_sumcheck_bind_eval_arbitrary(const Strategy& S, fr_t* base, size_t stride, size_t q, const fr_t& r,
                                         const Finalize& fin, size_t min_q, cudaStream_t st);
int sumcheck_max_blocks();

// ---- K3: batched cubic round evaluation (sumcheck.rs:49-93) ----
// A, B: ncirc device pointers each to 2*half elements; Ceq: 2*half elements. out = ncirc x 3 (e0,e2,e3).
void launch_sumcheck_eval_cubic(fr_t* const* d_A, fr_t* const* d_B, const fr_t* Ceq, int ncirc, size_t half,
                                const Finalize& fin, cudaStream_t st);

// What the prover runs (poly_kernels.cu): the same rounds with the batching coefficients of sumcheck.rs:95-97 folded
// in — out = 3 elements  sum_k coeff_k (e0, e2, e3)_k.  scale != 0: the arrays A_k are still unscaled in memory (the
// first evaluation and the first bind of a layer); the first bind stores coeff_k * A_k and later rounds use scale = 0.
struct CubicCoeffs {
  fr_t v[32];
};
void launch_sumcheck_eval_cubic_comb(fr_t* const* d_A, fr_t* const* d_B, const fr_t* Ceq, int ncirc, size_t half,
                                     const CubicCoeffs& cf, int scale, const Finalize& fin, cudaStream_t st);
// fused: bind A_k, B_k (in place) and eq (Cin -> Cout) with r, then evaluate the next round on the bound values;
// h = bound length (>= 2)
void launch_sumcheck_bind_eval_cubic_comb(fr_t* const* d_A, fr_t* const* d_B, const fr_t* Cin, fr_t* Cout, int ncirc, size_t h,
                                          const fr_t& r, const CubicCoeffs& cf, int scale, const Finalize& fin, cudaStream_t st);

// ---- K5: subtables (subtables/*.rs) ----
// tables_fr: nsub x M Montgomery elements; tables_u32: nsub x M raw values
void launch_materialize_subtables(const Strategy& S, fr_t* tables_fr, uint32_t* tables_u32, cudaStream_t st);
// E_k[j] = T_sub(k)[nz_dim(k)[j]] for k < alpha (subtables/mod.rs:78-92). nz: C x s (u32).
void launch_gather_lookup_polys(const Strategy& S, const fr_t* tables_fr, const uint32_t* tables_u32,
                                const uint32_t* nz, size_t s, fr_t* E_fr, size_t E_stride, uint32_t* E_u32,
                                cudaStream_t st);
// out[i] = F::from(in[i])  (dense_mlpoly.rs:263-269)
void launch_from_u32(const uint32_t* in, fr_t* out, size_t n, cudaStream_t st);
void launch_fill_zero(fr_t* out, size_t n, cudaStream_t st);

// ---- K7: supporting reductions ----
// out[k] = <P_k, eq>, P_k = base + k*stride, k < npolys, n elements each
void launch_multi_dot(const fr_t* base, size_t stride, int npolys, const fr_t* eq, size_t n, fr_t* partial,
                      fr_t* out, cudaStream_t st);
// sum_k eq[k] * g(E_1[k..]) (subtables/mod.rs:186-216)
void launch_sumcheck_claim(const Strategy& S, const fr_t* base, size_t stride, size_t n, fr_t* partial, fr_t* out,
                           cudaStream_t st);
// LZ[i] = sum_j L[j] Z[j*R_size + i] (dense_mlpoly.rs:183-207); partial: chunks x R_size scratch
void launch_bound(const fr_t* Z, const fr_t* L, size_t L_size, size_t R_size, fr_t* partial, fr_t* out,
                  cudaStream_t st);
int bound_max_chunks();
// the same two reductions over the u32 mirror of an INTEGER-valued polynomial (dim, read, final, E): 8 IMAD per term
// instead of a Montgomery product, 4 B read per element instead of 32 B, one reduction at the end
void launch_bound_u32(const uint32_t* Z, const fr_t* L, size_t L_size, size_t R_size, fr_t* partial, fr_t* out, cudaStream_t st);
void launch_multi_dot_u32(const uint32_t* base, size_t stride, int npolys, const fr_t* eq, size_t n, fr_t* partial, fr_t* out,
                          cudaStream_t st);
// Reed-Solomon fingerprints (memory_checking.rs:236-310).  init/final over M cells, read/write over s ops.
// M_local cells of this rank; local cell i = global address i*G + g; `table` is the full M-entry table
void launch_gp_fingerprints_mem(const fr_t* table, const fr_t* final_fr, size_t M_local, int G, int g,
                                const fr_t& gamma, const fr_t& tau, fr_t* out_init, fr_t* out_final, cudaStream_t st);
void launch_gp_fingerprints_ops(const fr_t* dim_fr, const fr_t* E_fr, const fr_t* read_fr, size_t s,
                                const fr_t& gamma, const fr_t& tau, fr_t* out_read, fr_t* out_write,
                                cudaStream_t st);
// product-tree layer (grand_product.rs:20-36): out[i] = in[i] * in[i + n_out], i < n_out
void launch_product_layer(const fr_t* in, fr_t* out, size_t n_out, cudaStream_t st);
// every product tree of one size N (contiguous layers, see poly_kernels.cu) + tagged publication of the two
// top-layer elements of tree t as values 2*(slot0 + t) + {0, 1}
struct TreePtrs {
  fr_t* p[32];
};
void launch_product_trees(const TreePtrs& trees, int ntrees, size_t N, int slot0, int stop_len, const Finalize& fin,
                          cudaStream_t st);
int product_trees_launches(size_t N);
// x_k[0] <- x_k[0] + r (x_k[1] - x_k[0]) for the n arrays x_k = d_AB[k]; results also published (Finalize)
void launch_bind_heads(fr_t* const* d_AB, int n, const fr_t& r, const Finalize& fin, cudaStream_t st);
// elementwise helpers for the Bulletproofs scalar folds (bullet.rs:125-130)
// a[i] <- a[i]*u + uinv*a[i+h];  b[i] <- b[i]*uinv + u*b[i+h]
void launch_fold_ab(fr_t* a, fr_t* b, size_t h, const fr_t& u, const fr_t& uinv, cudaStream_t st);
// out[0] = <a[0..h), b[h..2h)>, out[1] = <a[h..2h), b[0..h)>  (bullet.rs:78-79)
void launch_cross_inner_products(const fr_t* a, const fr_t* b, size_t h, fr_t* partial, fr_t* out, cudaStream_t st);
// w'[2t] = w[t]*uinv, w'[2t+1] = w[t]*u  (weights of the unfolded generators, see msm_kernels.cu)
void launch_expand_weights(const fr_t* w, fr_t* w_out, size_t n_in, const fr_t& u, const fr_t& uinv, cudaStream_t st);
// scalars for the L / R MSMs over the ORIGINAL generators: see prover.cu
void launch_bullet_round(const fr_t* a_in, const fr_t* b_in, const fr_t* w_in, fr_t* a_out, fr_t* b_out, fr_t* w_out, size_t n,
                         size_t m, int fold, const fr_t& u, const fr_t& uinv, const fr_t& blind_L, const fr_t& blind_R,
                         fr_t* s_out, uint32_t* cols_out, fr_t* partial, unsigned* counter, cudaStream_t st);
void launch_two_row_scalars(const fr_t* v, int scale, const fr_t& k, const fr_t& t00, const fr_t& t01, const fr_t& t10,
                            const fr_t& t11, size_t n, fr_t* out, cudaStream_t st);
void launch_bullet_scalars(const fr_t* a, const fr_t* w, size_t n_loc, size_t m, int G, int g, int a_rep, fr_t* sL,
                           fr_t* sR, cudaStream_t st);
void launch_scale(const fr_t* in, fr_t* out, size_t n, const fr_t& k, cudaStream_t st);

// ---- densify on the GPU (densify_kernels.cu; densified.rs:33-56): stable LSD radix sort by address ----
void densify_init_device();
bool densify_gpu_supported(size_t s, size_t log_m);
size_t densify_scratch_words(size_t s, int C, size_t log_m);
// The n x C index matrix on the device: element (k, dim) at p + k*row_stride + dim*col_stride (elements, >= 0), of one of
// four integer types (the values of LASSO_IDX_*).  bad (may be null): raised by the extract when an index is negative or
// >= m (that index is then counted as address 0).  bad_host (may be null, needs bad): pinned word the flag is copied
// to right after the extract, followed by a record of bad_ready, so the host can wait for the verdict alone.
enum { kDzU64 = 0, kDzI64 = 1, kDzU32 = 2, kDzI32 = 3 };
struct DzSource {
  const void* p = nullptr;
  int type = kDzU32;
  int64_t row_stride = 0, col_stride = 1;
  uint32_t* bad = nullptr;
  uint32_t* bad_host = nullptr;
  cudaEvent_t bad_ready = nullptr;
};
// All C dimensions at once; outputs are this rank's shards (rank g of G: accesses k = i*G + g, addresses a = i*G + g):
// dim_i at dim_loc + i*dim_stride, read_i at read_loc + i*read_stride, final_i likewise.
int launch_densify(const DzSource& src, size_t n, size_t s, int C, size_t log_m, int G, int g, uint32_t* scratch,
                   uint32_t* dim_loc, size_t dim_stride, uint32_t* read_loc, size_t read_stride, uint32_t* final_loc,
                   size_t final_stride, cudaStream_t st);

}  // namespace lb
