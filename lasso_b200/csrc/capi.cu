// lasso_b200 — extern "C" boundary (include/lasso_b200.h).  Plain pointers and sizes only; every entry
// point states the reference item it replaces in the header.
#include "../../include/lasso_b200.h"

#include "prover.cuh"

using namespace lb;

struct lasso_ctx {
  Ctx* c;
};
struct lasso_gens {
  Gens* g;
};
struct lasso_dense {
  Dense* d;
};

struct lasso_msm_job {
  Ctx* c = nullptr;
  size_t n = 0, n_pool = 0;
  DBuf<fq_t> bases;     // n_pool x (x, y) arkworks limbs
  DBuf<fr_t> scalars;   // n Montgomery scalars
  DBuf<pt_niels> niels; // n
  DBuf<fr_t> canon;     // n
  DBuf<uint8_t> scratch;
  DBuf<fq_t> out_ext;
  DBuf<uint32_t> raw;   // (G + 1) x 32 words: partial points of the ranks
  DBuf<pt_ext> naive_part;
  MsmLargePlan plan;    // of the last run
};

static thread_local std::string g_err;
static int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define LB_TRY try {
// every entry point that takes a context makes the context's device current first: a process may hold contexts on
// several GPUs, and kernel launches / allocations go to the CURRENT device
#define LB_TRY_CTX(h) \
  try {               \
    if (!(h) || !(h)->c) return fail(-1, "null context"); \
    LB_CUDA_CHECK(cudaSetDevice((h)->c->device));
#define LB_CATCH                                  \
  }                                               \
  catch (const std::exception& e) {               \
    return fail(-1, e.what());                    \
  }

static bool is_pow2(size_t x) { return x && !(x & (x - 1)); }
static constexpr size_t kMsmLargeMin = 1 << 14;  // below this the row kernels (c = 8, buckets in shared memory) win
static Strategy mkS(int kind, int C, int log_M, int log_R) { return Strategy{kind, C, log_M, log_R}; }

extern "C" {

const char* lasso_last_error(void) { return g_err.c_str(); }

int lasso_ctx_create(lasso_ctx** out, int device_id) {
  LB_TRY
  *out = nullptr;
  Ctx* c = ctx_create(device_id);
  *out = new lasso_ctx{c};
  return 0;
  LB_CATCH
}
void lasso_ctx_destroy(lasso_ctx* ctx) {
  if (!ctx) return;
  try {
    comm_destroy(ctx->c);
  } catch (...) {
  }
  ctx_destroy(ctx->c);
  delete ctx;
}
int lasso_comm_unique_id(uint8_t out[128]) {
  LB_TRY
  comm_unique_id(out);
  return 0;
  LB_CATCH
}
int lasso_ctx_init_comm(lasso_ctx* h, const uint8_t id[128], int rank, int world) {
  LB_TRY_CTX(h)
  comm_init(h->c, id, rank, world);
  return 0;
  LB_CATCH
}

int lasso_ctx_bind_host_threads(lasso_ctx* h) {
  if (!h || !h->c) return -1;
  return bind_host_threads(h->c->device, &h->c->helper_mask, &h->c->have_helper_mask);
}

int lasso_bind_top(lasso_ctx* h, uint64_t* Z, size_t len, const uint64_t r[4]) {
  LB_TRY_CTX(h)
  if (!is_pow2(len) || len < 2) return fail(LASSO_ERR_NOT_POW2, "bind_top: len must be a power of two >= 2");
  Ctx* c = h->c;
  DBuf<fr_t> d(c, len);
  LB_CUDA_CHECK(cudaMemcpyAsync(d.p, Z, len * 32, cudaMemcpyHostToDevice, c->st));
  fr_t rr;
  memcpy(rr.v, r, 32);
  launch_bind_top(d.p, 0, 1, len / 2, rr, c->st);
  g_launches++;
  LB_CUDA_CHECK(cudaMemcpyAsync(Z, d.p, (len / 2) * 32, cudaMemcpyDeviceToHost, c->st));
  c->sync();
  return 0;
  LB_CATCH
}
int lasso_bind_bot(lasso_ctx* h, uint64_t* Z, size_t len, const uint64_t r[4]) {
  LB_TRY_CTX(h)
  if (!is_pow2(len) || len < 2) return fail(LASSO_ERR_NOT_POW2, "bind_bot: len must be a power of two >= 2");
  Ctx* c = h->c;
  DBuf<fr_t> d(c, len), o(c, len / 2);
  LB_CUDA_CHECK(cudaMemcpyAsync(d.p, Z, len * 32, cudaMemcpyHostToDevice, c->st));
  fr_t rr;
  memcpy(rr.v, r, 32);
  launch_bind_bot(d.p, o.p, len / 2, rr, c->st);
  g_launches++;
  LB_CUDA_CHECK(cudaMemcpyAsync(Z, o.p, (len / 2) * 32, cudaMemcpyDeviceToHost, c->st));
  c->sync();
  return 0;
  LB_CATCH
}
int lasso_eq_evals(lasso_ctx* h, const uint64_t* r, int ell, uint64_t* out) {
  LB_TRY_CTX(h)
  if (ell < 0 || ell > 28) return fail(LASSO_ERR_LENGTH, "eq_evals: 0 <= ell <= 28");
  Ctx* c = h->c;
  FrVec rv;
  for (int i = 0; i < ell; i++) memcpy(rv.v[i].v, r + 4 * i, 32);
  size_t n = (size_t)1 << ell;
  DBuf<fr_t> d(c, n);
  launch_eq_evals(rv, ell, d.p, c->d_eq_scratch, c->st);
  g_launches += ell <= 11 ? 1 : (ell <= 22 ? 3 : 5);
  LB_CUDA_CHECK(cudaMemcpyAsync(out, d.p, n * 32, cudaMemcpyDeviceToHost, c->st));
  c->sync();
  return 0;
  LB_CATCH
}
int lasso_sumcheck_round_arbitrary(lasso_ctx* h, int strategy, int C, int log_M, int log_R,
                                   const uint64_t* const* polys, size_t len, uint64_t* evals_out) {
  LB_TRY_CTX(h)
  Strategy S = mkS(strategy, C, log_M, log_R);
  if (!S.valid()) return fail(LASSO_ERR_STRATEGY, "unsupported strategy parameters");
  if (!is_pow2(len) || len < 2) return fail(LASSO_ERR_NOT_POW2, "len must be a power of two >= 2");
  Ctx* c = h->c;
  int np = S.num_memories() + 1, npts = S.sumcheck_poly_degree() + 1;
  DBuf<fr_t> d(c, (size_t)np * len);
  for (int k = 0; k < np; k++)
    LB_CUDA_CHECK(cudaMemcpyAsync(d.p + (size_t)k * len, polys[k], len * 32, cudaMemcpyHostToDevice, c->st));
  Finalize f = c->fin_begin();
  f.pub.ndst = 0;  // plain device result + copy on this entry point
  launch_sumcheck_eval_arbitrary(S, d.p, len, len / 2, f, c->st);
  g_launches += 1;
  c->d2h(evals_out, c->d_small, (size_t)npts * 32);
  return 0;
  LB_CATCH
}
int lasso_sumcheck_bind_round_arbitrary(lasso_ctx* h, int strategy, int C, int log_M, int log_R, uint64_t* const* polys,
                                        size_t len, const uint64_t r[4], uint64_t* evals_out) {
  LB_TRY_CTX(h)
  Strategy S = mkS(strategy, C, log_M, log_R);
  if (!S.valid()) return fail(LASSO_ERR_STRATEGY, "unsupported strategy parameters");
  if (!is_pow2(len) || len < 4) return fail(LASSO_ERR_NOT_POW2, "len must be a power of two >= 4");
  Ctx* c = h->c;
  const int np = S.num_memories() + 1, npts = S.sumcheck_poly_degree() + 1;
  DBuf<fr_t> d(c, (size_t)np * len);
  for (int k = 0; k < np; k++)
    LB_CUDA_CHECK(cudaMemcpyAsync(d.p + (size_t)k * len, polys[k], len * 32, cudaMemcpyHostToDevice, c->st));
  fr_t rr;
  memcpy(&rr, r, 32);
  Finalize f = c->fin_begin();
  f.pub.ndst = 0;  // plain device result + copy on this entry point
  if (!launch_sumcheck_bind_eval_arbitrary(S, d.p, len, len / 4, rr, f, 1, c->st)) {
    launch_bind_top(d.p, len, np, len / 2, rr, c->st);
    launch_sumcheck_eval_arbitrary(S, d.p, len, len / 4, f, c->st);
    g_launches += 1;
  }
  g_launches += 1;
  c->d2h(evals_out, c->d_small, (size_t)npts * 32);
  for (int k = 0; k < np; k++) c->d2h(polys[k], d.p + (size_t)k * len, (len / 2) * 32);
  return 0;
  LB_CATCH
}
int lasso_sumcheck_round_cubic(lasso_ctx* h, int n_circuits, const uint64_t* const* A, const uint64_t* const* B,
                               const uint64_t* Ceq, size_t len, uint64_t* out) {
  LB_TRY_CTX(h)
  if (!is_pow2(len) || len < 2) return fail(LASSO_ERR_NOT_POW2, "len must be a power of two >= 2");
  if (n_circuits < 1 || n_circuits > 512) return fail(LASSO_ERR_LENGTH, "1 <= n_circuits <= 512");
  Ctx* c = h->c;
  DBuf<fr_t> dA(c, (size_t)n_circuits * len), dB(c, (size_t)n_circuits * len), dC(c, len);
  DBuf<fr_t*> pA(c, n_circuits), pB(c, n_circuits);
  std::vector<fr_t*> hA(n_circuits), hB(n_circuits);
  for (int k = 0; k < n_circuits; k++) {
    hA[k] = dA.p + (size_t)k * len;
    hB[k] = dB.p + (size_t)k * len;
    LB_CUDA_CHECK(cudaMemcpyAsync(hA[k], A[k], len * 32, cudaMemcpyHostToDevice, c->st));
    LB_CUDA_CHECK(cudaMemcpyAsync(hB[k], B[k], len * 32, cudaMemcpyHostToDevice, c->st));
  }
  LB_CUDA_CHECK(cudaMemcpyAsync(dC.p, Ceq, len * 32, cudaMemcpyHostToDevice, c->st));
  LB_CUDA_CHECK(cudaMemcpyAsync(pA.p, hA.data(), n_circuits * sizeof(fr_t*), cudaMemcpyHostToDevice, c->st));
  LB_CUDA_CHECK(cudaMemcpyAsync(pB.p, hB.data(), n_circuits * sizeof(fr_t*), cudaMemcpyHostToDevice, c->st));
  Finalize f = c->fin_begin();
  f.pub.ndst = 0;
  launch_sumcheck_eval_cubic(pA.p, pB.p, dC.p, n_circuits, len / 2, f, c->st);
  g_launches += 1;
  c->d2h(out, c->d_small, (size_t)n_circuits * 3 * 32);
  return 0;
  LB_CATCH
}
int lasso_materialize_subtables(lasso_ctx* h, int strategy, int C, int log_M, int log_R, uint64_t* const* tables_out) {
  LB_TRY_CTX(h)
  Strategy S = mkS(strategy, C, log_M, log_R);
  if (!S.valid()) return fail(LASSO_ERR_STRATEGY, "unsupported strategy parameters");
  Ctx* c = h->c;
  size_t M = (size_t)S.M();
  DBuf<fr_t> t(c, M * S.num_subtables());
  launch_materialize_subtables(S, t.p, nullptr, c->st);
  g_launches++;
  for (int k = 0; k < S.num_subtables(); k++)
    LB_CUDA_CHECK(cudaMemcpyAsync(tables_out[k], t.p + (size_t)k * M, M * 32, cudaMemcpyDeviceToHost, c->st));
  c->sync();
  return 0;
  LB_CATCH
}
int lasso_gather_lookup_polys(lasso_ctx* h, int strategy, int C, int log_M, int log_R, const uint64_t* const* nz,
                              size_t s, uint64_t* const* E_out) {
  LB_TRY_CTX(h)
  Strategy S = mkS(strategy, C, log_M, log_R);
  if (!S.valid()) return fail(LASSO_ERR_STRATEGY, "unsupported strategy parameters");
  Ctx* c = h->c;
  size_t M = (size_t)S.M();
  std::vector<uint32_t> idx((size_t)C * s);
  for (int d = 0; d < C; d++)
    for (size_t j = 0; j < s; j++) {
      if (nz[d][j] >= M) return fail(LASSO_ERR_INDEX_RANGE, "lookup index out of range");
      idx[(size_t)d * s + j] = (uint32_t)nz[d][j];
    }
  DBuf<fr_t> t(c, M * S.num_subtables()), E(c, (size_t)S.num_memories() * s);
  DBuf<uint32_t> dn(c, (size_t)C * s);
  LB_CUDA_CHECK(cudaMemcpyAsync(dn.p, idx.data(), idx.size() * 4, cudaMemcpyHostToDevice, c->st));
  launch_materialize_subtables(S, t.p, nullptr, c->st);
  launch_gather_lookup_polys(S, t.p, nullptr, dn.p, s, E.p, s, nullptr, c->st);
  g_launches += 2;
  for (int k = 0; k < S.num_memories(); k++)
    LB_CUDA_CHECK(cudaMemcpyAsync(E_out[k], E.p + (size_t)k * s, s * 32, cudaMemcpyDeviceToHost, c->st));
  c->sync();
  return 0;
  LB_CATCH
}

// shared by lasso_msm / lasso_commit_rows: variable bases (window-0 table only), Montgomery scalars
static void msm_variable_base(Ctx* c, const uint64_t* bases_affine, size_t nbases, const uint64_t* scalars, size_t nrows,
                              size_t ncols, uint64_t* out_ext) {
  DBuf<fq_t> db(c, nbases * 2);
  DBuf<pt_niels> tab(c, nbases);
  DBuf<fr_t> sc(c, nrows * ncols), canon(c, nrows * ncols);
  LB_CUDA_CHECK(cudaMemcpyAsync(db.p, bases_affine, nbases * 64, cudaMemcpyHostToDevice, c->st));
  LB_CUDA_CHECK(cudaMemcpyAsync(sc.p, scalars, nrows * ncols * 32, cudaMemcpyHostToDevice, c->st));
  launch_build_table(db.p, nbases, tab.p, nbases, 1, c->st);
  LB_CUDA_CHECK(cudaMemsetAsync(c->d_flag, 0, 4, c->st));
  launch_canonicalize(sc.p, canon.p, nrows * ncols, c->d_flag, c->st);
  unsigned max_bits = 0;
  c->d2h(&max_bits, c->d_flag, 4);
  // the reference's small-scalar shortcut (msm/mod.rs:95-106) only changes the schedule, not the result;
  // here the window count simply follows the widest scalar
  int nw = msm_windows_for_bits(max_bits);
  if (nw > kMsmFullWindows) nw = kMsmFullWindows;
  DBuf<pt_ext> part(c, msm_partials_count((int)nrows, (int)ncols, nw));
  DBuf<fq_t> oe(c, nrows * 4);
  if (c->world == 1) {
    launch_msm_rows(tab.p, nbases, 0, canon.p, 8, ncols, (int)nrows, (int)ncols, nw, 1, 0, part.p, oe.p, nullptr, nullptr, c->st);
    g_launches += 4;
  } else {
    // collective: every rank passed ITS shard of the terms; partial points are all-gathered and added
    // ("final bucket-sum reduce over NVLink" = gather-then-add, group addition is not an NCCL reduction)
    DBuf<uint32_t> raw(c, (size_t)(c->world + 1) * nrows * 32);
    uint32_t* mine = raw.p + (size_t)c->world * nrows * 32;
    launch_msm_rows(tab.p, nbases, 0, canon.p, 8, ncols, (int)nrows, (int)ncols, nw, 1, 0, part.p, nullptr, nullptr, mine, c->st);
    comm_allgather(c, mine, raw.p, nrows * 128);
    launch_sum_raw_points(raw.p, c->world, (int)nrows, nullptr, nullptr, oe.p, c->st);
    g_launches += 5;
  }
  LB_CUDA_CHECK(cudaMemcpyAsync(out_ext, oe.p, nrows * 128, cudaMemcpyDeviceToHost, c->st));
  c->sync();
}
// ---- one large MSM on device-resident inputs (msm_large.cu)
static lasso_msm_job* msm_job_make(Ctx* c, const uint64_t* bases_affine, size_t n_pool, const uint64_t* scalars, size_t n) {
  std::unique_ptr<lasso_msm_job> j(new lasso_msm_job());
  j->c = c;
  j->n = n;
  j->n_pool = n_pool;
  j->bases.alloc(c, n_pool * 2);
  j->scalars.alloc(c, n);
  j->niels.alloc(c, n);
  j->canon.alloc(c, n);
  j->scratch.alloc(c, msm_large_scratch_bytes(msm_large_plan(n, 253)));
  j->out_ext.alloc(c, 4);
  j->raw.alloc(c, (size_t)(c->world + 1) * 32);
  LB_CUDA_CHECK(cudaMemcpyAsync(j->bases.p, bases_affine, n_pool * 64, cudaMemcpyHostToDevice, c->st));
  LB_CUDA_CHECK(cudaMemcpyAsync(j->scalars.p, scalars, n * 32, cudaMemcpyHostToDevice, c->st));
  c->sync();
  return j.release();
}
// one MSM: prep (canonical scalars, niels bases, widest scalar) -> plan -> Pippenger; sharded: every rank's partial
// point is all-gathered and added ("final bucket-sum reduce over NVLink" = gather-then-add)
static void msm_job_once(lasso_msm_job* j) {
  Ctx* c = j->c;
  LB_CUDA_CHECK(cudaMemsetAsync(c->d_flag, 0, 4, c->st));
  launch_msm_large_prep(j->bases.p, j->scalars.p, j->n, j->n_pool == j->n ? 0 : j->n_pool, j->niels.p, j->canon.p, c->d_flag, c->st);
  unsigned max_bits = 0;
  c->d2h(&max_bits, c->d_flag, 4);
  // the reference's small-scalar shortcut (msm/mod.rs:95-106) only changes the schedule, not the result: here the
  // window count simply follows the widest scalar
  j->plan = msm_large_plan(j->n, max_bits);
  if (c->world == 1) {
    g_launches += 2 + launch_msm_large(j->plan, j->niels.p, j->canon.p, j->scratch.p, j->out_ext.p, nullptr, c->st);
    return;
  }
  uint32_t* mine = j->raw.p + (size_t)c->world * 32;
  g_launches += 2 + launch_msm_large(j->plan, j->niels.p, j->canon.p, j->scratch.p, nullptr, mine, c->st);
  comm_allgather(c, mine, j->raw.p, 128);
  launch_sum_raw_points(j->raw.p, c->world, 1, nullptr, nullptr, j->out_ext.p, c->st);
  g_launches += 1;
}
int lasso_msm_plan_info(size_t n, unsigned max_bits, int out[16]) {
  LB_TRY
  if (n == 0) return fail(LASSO_ERR_LENGTH, "msm plan: n >= 1");
  const MsmLargePlan p = msm_large_plan(n, max_bits);
  for (int i = 0; i < 16; i++) out[i] = 0;
  out[0] = p.c;
  out[1] = p.nw;
  out[2] = p.nbits;
  out[3] = (int)p.NB;
  out[4] = (int)p.S;
  out[5] = p.nlev;
  for (int k = 0; k < p.nlev && k < 8; k++) out[6 + k] = (int)p.lev_L[k];
  return 0;
  LB_CATCH
}
int lasso_msm_job_create(lasso_ctx* h, const uint64_t* bases_affine, size_t n_pool, const uint64_t* scalars, size_t n,
                         lasso_msm_job** out) {
  LB_TRY_CTX(h)
  *out = nullptr;
  if (n == 0 || n >= ((size_t)1 << 31) || n_pool == 0 || n_pool > n) return fail(LASSO_ERR_LENGTH, "msm job: 1 <= n_pool <= n < 2^31");
  *out = msm_job_make(h->c, bases_affine, n_pool, scalars, n);
  return 0;
  LB_CATCH
}
int lasso_msm_job_run(lasso_ctx* h, lasso_msm_job* j, int iters, double* avg_ms, uint64_t out_xytz[16], int info[8]) {
  LB_TRY_CTX(h)
  if (!j || j->c != h->c || iters < 1) return fail(LASSO_ERR_LENGTH, "msm job: bad arguments");
  Ctx* c = h->c;
  cudaEvent_t e0, e1;
  LB_CUDA_CHECK(cudaEventCreate(&e0));
  LB_CUDA_CHECK(cudaEventCreate(&e1));
  LB_CUDA_CHECK(cudaEventRecord(e0, c->st));
  for (int i = 0; i < iters; i++) msm_job_once(j);
  LB_CUDA_CHECK(cudaEventRecord(e1, c->st));
  LB_CUDA_CHECK(cudaEventSynchronize(e1));
  float ms = 0;
  LB_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (avg_ms) *avg_ms = ms / iters;
  if (out_xytz) {
    LB_CUDA_CHECK(cudaMemcpyAsync(out_xytz, j->out_ext.p, 128, cudaMemcpyDeviceToHost, c->st));
    c->sync();
  }
  if (info) {
    info[0] = j->plan.c;
    info[1] = j->plan.nw;
    info[2] = j->plan.nbits;
    info[3] = (int)j->plan.S;
    info[4] = (int)j->plan.lev_L[0];
    info[5] = j->plan.nlev;
    info[6] = c->world;
    info[7] = 0;
  }
  return 0;
  LB_CATCH
}
int lasso_msm_job_naive(lasso_ctx* h, lasso_msm_job* j, uint64_t out_xytz[16]) {
  LB_TRY_CTX(h)
  if (!j || j->c != h->c) return fail(LASSO_ERR_LENGTH, "msm job: bad arguments");
  Ctx* c = h->c;
  if (c->world > 1) return fail(LASSO_ERR_LENGTH, "msm job: the naive cross-check is single-GPU");
  if (!j->naive_part.p) j->naive_part.alloc(c, (size_t)kNumSMs * 8);
  launch_msm_naive(j->bases.p, j->scalars.p, j->n, j->n_pool == j->n ? 0 : j->n_pool, j->naive_part.p, j->out_ext.p, c->st);
  g_launches += 2;
  LB_CUDA_CHECK(cudaMemcpyAsync(out_xytz, j->out_ext.p, 128, cudaMemcpyDeviceToHost, c->st));
  c->sync();
  return 0;
  LB_CATCH
}
void lasso_msm_job_destroy(lasso_msm_job* j) {
  if (!j) return;
  cudaSetDevice(j->c->device);
  delete j;
}

int lasso_msm(lasso_ctx* h, const uint64_t* bases_affine, const uint64_t* scalars, size_t n, uint64_t out_xytz[16]) {
  LB_TRY_CTX(h)
  if (n == 0 || n > (1u << 30)) return fail(LASSO_ERR_LENGTH, "msm: 1 <= n <= 2^30");
  if (n >= kMsmLargeMin) {  // one large MSM: the large-window Pippenger (msm_large.cu); collective when sharded
    std::unique_ptr<lasso_msm_job> j(msm_job_make(h->c, bases_affine, n, scalars, n));
    msm_job_once(j.get());
    LB_CUDA_CHECK(cudaMemcpyAsync(out_xytz, j->out_ext.p, 128, cudaMemcpyDeviceToHost, h->c->st));
    h->c->sync();
    return 0;
  }
  msm_variable_base(h->c, bases_affine, n, scalars, 1, n, out_xytz);
  return 0;
  LB_CATCH
}
int lasso_commit_rows(lasso_ctx* h, const uint64_t* gens_affine, const uint64_t* Z, size_t L_size, size_t R_size,
                      uint64_t* out_points) {
  LB_TRY_CTX(h)
  if (!L_size || !R_size) return fail(LASSO_ERR_LENGTH, "commit_rows: empty matrix");
  // blind = 0 on this path, so the trailing generator h contributes nothing (commitments.rs:89-92)
  msm_variable_base(h->c, gens_affine, R_size, Z, L_size, R_size, out_points);
  return 0;
  LB_CATCH
}

size_t lasso_gens_points_needed(size_t c, size_t s, size_t num_memories, size_t log_m) {
  return gens_points_needed(c, s, num_memories, log_m);
}
int lasso_sample_generators(const char* label, size_t count, uint64_t* out_affine) {
  LB_TRY
  sample_generators(label, count, out_affine);
  return 0;
  LB_CATCH
}
int lasso_gens_create(lasso_ctx* h, const uint64_t* stream_affine, size_t n_points, size_t c, size_t s,
                      size_t num_memories, size_t log_m, lasso_gens** out) {
  LB_TRY_CTX(h)
  *out = nullptr;
  if (!is_pow2(s)) return fail(LASSO_ERR_NOT_POW2, "s must be a power of two");
  Gens* g = gens_create(h->c, stream_affine, n_points, c, s, num_memories, log_m);
  if (!g) return fail(LASSO_ERR_GENS, "generator stream shorter than lasso_gens_points_needed()");
  *out = new lasso_gens{g};
  return 0;
  LB_CATCH
}
void lasso_gens_destroy(lasso_gens* g) {
  if (!g) return;
  delete g->g;
  delete g;
}

int lasso_densify(lasso_ctx* h, const uint64_t* indices, size_t n_lookups, size_t C, size_t log_m, lasso_dense** out) {
  LB_TRY_CTX(h)
  *out = nullptr;
  auto t0 = std::chrono::steady_clock::now();
  int err = 0;
  Dense* d = densify(h->c, indices, n_lookups, C, log_m, &err);
  if (!d) return fail(err == 3 ? LASSO_ERR_INDEX_RANGE : LASSO_ERR_STRATEGY, "densify: invalid input");
  h->c->t_densify_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *out = new lasso_dense{d};
  return 0;
  LB_CATCH
}
int lasso_densify_device(lasso_ctx* h, const void* indices, int dtype, size_t n_lookups, size_t C, int64_t row_stride,
                         int64_t col_stride, size_t log_m, void* cuda_stream, lasso_dense** out) {
  LB_TRY_CTX(h)
  *out = nullptr;
  auto t0 = std::chrono::steady_clock::now();
  int err = 0;
  Dense* d = densify_device(h->c, indices, dtype, n_lookups, C, row_stride, col_stride, log_m,
                            static_cast<cudaStream_t>(cuda_stream), &err);
  if (!d)
    return err == 3 ? fail(LASSO_ERR_INDEX_RANGE, "densify_device: lookup index negative or >= m")
                    : fail(LASSO_ERR_STRATEGY, "densify_device: invalid shape, strides or index type");
  h->c->t_densify_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *out = new lasso_dense{d};
  return 0;
  LB_CATCH
}
void lasso_dense_destroy(lasso_dense* d) {
  if (!d) return;
  delete d->d;
  delete d;
}
size_t lasso_dense_s(const lasso_dense* d) { return d->d->s; }
size_t lasso_dense_read(lasso_ctx* h, const lasso_dense* dd, int which, uint64_t* out, size_t cap) {
  try {
    const Dense& d = *dd->d;
    Ctx* c = h->c;
    LB_CUDA_CHECK(cudaSetDevice(c->device));
    if (c->world > 1) {  // the arrays hold this rank's low-bit shard only: the field views below do not apply
      g_err = "lasso_dense_read is not available on a sharded context";
      return 0;
    }
    size_t n = 0;
    if (which == 0) {
      n = d.C * d.s;
      if (n > cap) return 0;
      std::vector<uint32_t> tmp(n);
      c->d2h(tmp.data(), d.d_l_u32.p, n * 4);
      for (size_t i = 0; i < n; i++) out[i] = tmp[i];
      return n;
    }
    const fr_t* src = nullptr;
    switch (which) {
      case 1: src = d.d_l_fr.p; n = d.C * d.s; break;
      case 2: src = d.d_l_fr.p + d.C * d.s; n = d.C * d.s; break;
      case 3: src = d.d_m_fr.p; n = d.C * d.m; break;
      case 4: src = d.d_l_fr.p; n = (size_t)1 << d.nv_l; break;
      case 5: src = d.d_m_fr.p; n = (size_t)1 << d.nv_m; break;
      default: return 0;
    }
    if (n > cap) return 0;
    c->d2h(out, src, n * 32);
    return n;
  } catch (const std::exception& e) {
    g_err = e.what();
    return 0;
  }
}

int lasso_commit(lasso_ctx* h, const lasso_dense* d, const lasso_gens* g, uint8_t* out, size_t cap, size_t* out_len) {
  LB_TRY_CTX(h)
  auto t0 = std::chrono::steady_clock::now();
  std::vector<uint8_t> b = commit(h->c, *d->d, *g->g);
  h->c->t_commit_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *out_len = b.size();
  if (b.size() > cap) return fail(LASSO_ERR_LENGTH, "commit: output buffer too small");
  memcpy(out, b.data(), b.size());
  return 0;
  LB_CATCH
}

int lasso_prove(lasso_ctx* h, int strategy, int log_R, lasso_dense* d, const uint64_t* r, size_t r_len,
                const lasso_gens* g, const char* transcript_label, const char* tape_label, const uint64_t tape_seed[4],
                uint8_t* proof_out, size_t proof_cap, size_t* proof_len, uint64_t* challenges_out,
                size_t challenges_cap, size_t* n_challenges) {
  LB_TRY_CTX(h)
  Strategy S = mkS(strategy, (int)d->d->C, (int)d->d->log_m, log_R);
  if (!S.valid()) return fail(LASSO_ERR_STRATEGY, "unsupported strategy parameters");
  // assert_eq!(r.len(), log2(dense.s))  surge.rs:131
  if (r_len != log2_exact_or_ceil(d->d->s)) return fail(LASSO_ERR_LENGTH, "r.len() != log2(s)");
  std::vector<fr_t> rv(r_len);
  for (size_t i = 0; i < r_len; i++) memcpy(rv[i].v, r + 4 * i, 32);
  fr_t seed;
  memcpy(seed.v, tape_seed, 32);
  std::vector<fr_t> trace;
  auto t0 = std::chrono::steady_clock::now();
  std::vector<uint8_t> b;
  try {
    b = prove(h->c, S, *d->d, rv, *g->g, transcript_label, tape_label, seed, &trace);
  } catch (const std::runtime_error& e) {
    if (std::string(e.what()).find("multiset") != std::string::npos) return fail(LASSO_ERR_MULTISET, e.what());
    throw;
  }
  h->c->t_prove_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  *proof_len = b.size();
  if (n_challenges) *n_challenges = trace.size();
  if (challenges_out)
    for (size_t i = 0; i < trace.size() && i < challenges_cap; i++) memcpy(challenges_out + 4 * i, trace[i].v, 32);
  if (b.size() > proof_cap) return fail(LASSO_ERR_LENGTH, "prove: output buffer too small");
  memcpy(proof_out, b.data(), b.size());
  return 0;
  LB_CATCH
}

unsigned long long lasso_launch_count(const lasso_ctx*) { return g_launches.load(); }
void lasso_last_timings(const lasso_ctx* h, double out_ms[3]) {
  out_ms[0] = h->c->t_densify_ms;
  out_ms[1] = h->c->t_commit_ms;
  out_ms[2] = h->c->t_prove_ms;
}
size_t lasso_spans(const lasso_ctx* h, char* buf, size_t cap) {
  std::string s;
  for (auto& kv : h->c->spans) s += kv.first + "=" + std::to_string(kv.second) + ";";
  if (buf && cap) {
    size_t n = std::min(cap - 1, s.size());
    memcpy(buf, s.data(), n);
    buf[n] = 0;
  }
  h->c->spans.clear();
  return s.size();
}

int lasso_bench_bind(lasso_ctx* h, size_t len, int npolys, int iters, double* avg_ms) {
  LB_TRY_CTX(h)
  if (!is_pow2(len) || len < 2 || npolys < 1) return fail(LASSO_ERR_NOT_POW2, "bench_bind: bad shape");
  Ctx* c = h->c;
  DBuf<fr_t> d(c, len * npolys);
  // fill with pseudo-random canonical residues: eq table of a fixed point, replicated
  FrVec rv;
  int ell = 0;
  while (((size_t)1 << ell) < len) ell++;
  for (int i = 0; i < ell; i++) rv.v[i] = fr_from_u64(0x9e3779b97f4a7c15ull * (i + 1));
  for (int k = 0; k < npolys; k++) launch_eq_evals(rv, ell, d.p + (size_t)k * len, c->d_eq_scratch, c->st);
  fr_t r = fr_from_u64(0xdeadbeefcafef00dull);
  cudaEvent_t e0, e1;
  LB_CUDA_CHECK(cudaEventCreate(&e0));
  LB_CUDA_CHECK(cudaEventCreate(&e1));
  for (int w = 0; w < 3; w++) launch_bind_top(d.p, len, npolys, len / 2, r, c->st);
  c->sync();
  LB_CUDA_CHECK(cudaEventRecord(e0, c->st));
  for (int i = 0; i < iters; i++) launch_bind_top(d.p, len, npolys, len / 2, r, c->st);
  LB_CUDA_CHECK(cudaEventRecord(e1, c->st));
  LB_CUDA_CHECK(cudaEventSynchronize(e1));
  g_launches += iters + 3;
  float ms = 0;
  LB_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
  *avg_ms = ms / iters;
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return 0;
  LB_CATCH
}

}  // extern "C"
