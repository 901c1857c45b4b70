// lasso_b200 — host-side prover objects: context, device buffers, generator tables, the
// densified representation and the proof byte writer.  The prover logic is in prover.cu.
#pragma once
#include <sched.h>

#include <atomic>
#include <chrono>
#include <map>
#include <memory>
#include <vector>

#include "host_transcript.hpp"
#include "kernels.cuh"
#include "msm.cuh"

namespace lb {

extern std::atomic<unsigned long long> g_launches;  // kernels launched by this process (bench.py's gpu_launches)

struct Ctx {
  int device = 0;
  cudaStream_t st = nullptr;
  uint8_t* h_pin = nullptr;  // pinned staging for small device->host results
  size_t h_pin_bytes = 0;
  fr_t* d_partial = nullptr;  // block partial sums / bound chunks
  size_t partial_elems = 0;
  fr_t* d_small = nullptr;  // small results (<= 64K elements)
  size_t small_elems = 0;
  fr_t* d_eq_scratch = nullptr;
  unsigned* d_flag = nullptr;
  uint32_t* h_stage = nullptr;  // pinned staging for the densified integer arrays (grown on demand, reused)
  size_t h_stage_elems = 0;
  uint32_t* stage(size_t elems) {
    if (elems > h_stage_elems) {
      if (h_stage) cudaFreeHost(h_stage);
      h_stage = nullptr;
      h_stage_elems = 0;  // a failed allocation below must not leave a stale size behind
      LB_CUDA_CHECK(cudaMallocHost((void**)&h_stage, elems * sizeof(uint32_t)));
      h_stage_elems = elems;
    }
    return h_stage;
  }
  // ---- single proof sharded over `world` GPUs (comm.cu); world == 1: everything below is inert
  int world = 1, rank = 0, lg_world = 0;
  void* xchg = nullptr;  // comm.cu: shared host segments + peer exchange buffers
  bool h_pub_owned = false;
  fr_t* d_gather = nullptr;  // all-gather landing zone
  size_t gather_elems = 0;
  double t_densify_ms = 0, t_commit_ms = 0, t_prove_ms = 0;
  std::map<std::string, double> spans;  // filled when LASSO_B200_SPANS=1 (forces syncs)
  bool span_sync = false;

  void sync() { LB_CUDA_CHECK(cudaStreamSynchronize(st)); }
  // Small results (<= 4 KiB) that are not round messages: a one-warp kernel copies the result into mapped pinned
  // host memory and then raises a sequence flag (system-scope fence); the host spins on the flag.  ~10-15 us
  // cheaper than cudaMemcpyAsync + cudaStreamSynchronize.
  uint32_t* h_mapped = nullptr;  // [0..1024) payload words, [1024] flag
  uint32_t* d_mapped = nullptr;
  uint32_t mapped_seq = 0;
  static constexpr size_t kMappedBytes = 8192;
  // Tagged publication of round messages and MSM points (common.cuh PubDst): this process's receive buffer
  // [writer][region][element][kPubSlotWords] and the device view of every reader's buffer (world == 1: only its
  // own, plain cudaHostAlloc; world > 1: shared pinned host segments mapped by every process, comm.cu)
  unsigned long long* h_pub = nullptr;
  unsigned long long* d_pub_reader[kPubMaxReaders] = {};
  uint32_t pub_seq = 0;
  static constexpr size_t kPubBytes = (size_t)kPubMaxReaders * kPubRegions * kPubElems * kPubSlotWords * 8;  // 1 MiB
  cudaEvent_t ev_aux = nullptr;  // marks a device->host copy that overlaps later launches on the same stream
  cudaEvent_t ev_stage = nullptr;  // recorded after the last upload out of h_stage (the buffer is reused by the next densify)
  bool stage_busy = false;
  cudaEvent_t ev_input = nullptr;  // recorded on the caller's stream: densify_device waits there for its input's producer
  // host-thread placement (bind_host_threads): the CPUs the library's helper threads may use
  cpu_set_t helper_mask;
  bool have_helper_mask = false;
  void helper_thread_enter() const {
    if (have_helper_mask) sched_setaffinity(0, sizeof helper_mask, &helper_mask);
  }
  void d2h_small(void* dst, const void* src, size_t bytes);  // prover.cu
  void wait_flag(uint32_t seq);                               // prover.cu
  // next message: `all` = every rank stores into every reader's buffer and the readers add the G residues
  // (the per-round exchange of a sharded proof); otherwise the message goes to this process only
  PubDst pub_begin(bool all) {
    PubDst p;
    p.ndst = 0;
    p.tag = 0;
    p.region = 0;
    p.all = 0;
    for (int i = 0; i < kPubMaxReaders; i++) p.dst[i] = nullptr;
    if (!h_pub) return p;
    const uint32_t seq = pub_seq++;
    p.region = (int)(seq % kPubRegions);
    p.tag = 1 + seq % kPubTagMod;
    p.all = (all && world > 1) ? 1 : 0;
    const size_t off = ((size_t)rank * kPubRegions + p.region) * kPubElems * kPubSlotWords;
    if (p.all) {
      for (int r = 0; r < world; r++) p.dst[p.ndst++] = d_pub_reader[r] + off;
    } else {
      p.dst[p.ndst++] = d_pub_reader[rank] + off;
    }
    return p;
  }
  // count elements of 8 x u32 words from one writer's region; blocks until every word carries the tag
  void pub_wait_raw(const PubDst& p, int writer, int count, uint32_t* out);  // prover.cu
  // a round message produced by a single launch (common.cuh Finalize): results land in d_small and directly in
  // the mapped host buffer(s); reduce = sum over the ranks of a sharded proof
  Finalize fin_begin(bool reduce = false) {
    Finalize f;
    f.partial = d_partial;
    f.counter = d_flag + 4;
    f.out_dev = d_small;
    f.pub = pub_begin(reduce);
    return f;
  }
  void fin_wait(const Finalize& f, fr_t* dst, int count);  // prover.cu (adds the residues of all ranks when f.pub.all)
  // npoints x (X, Y, Z) canonical Fq limbs published by msm_finish_quad_kernel
  void wait_points(const PubDst& p, int npoints, uint32_t* xyz /* npoints x 24 words */);
  // device -> host through the pinned buffer (small) or directly (large)
  void d2h(void* dst, const void* src, size_t bytes) {
    if (bytes <= 4096 && h_mapped) {
      d2h_small(dst, src, bytes);
      return;
    }
    if (bytes <= h_pin_bytes) {
      LB_CUDA_CHECK(cudaMemcpyAsync(h_pin, src, bytes, cudaMemcpyDeviceToHost, st));
      sync();
      memcpy(dst, h_pin, bytes);
    } else {
      LB_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st));
      sync();
    }
  }
  void h2d(void* dst, const void* src, size_t bytes) {
    LB_CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
    sync();  // the source may be a stack / pageable buffer
  }
};

// While helper threads are being CREATED the calling thread widens its own affinity to the helper CPUs: a new thread
// inherits its creator's mask, and a creator pinned to one core that goes on to spin there would leave its children
// waiting for that very core before they can even move themselves (milliseconds).  Restored on scope exit.
struct HelperSpawnScope {
  cpu_set_t saved;
  bool active = false;
  HelperSpawnScope(const Ctx* c, bool spawning) {
    if (spawning && c->have_helper_mask && sched_getaffinity(0, sizeof saved, &saved) == 0)
      active = sched_setaffinity(0, sizeof c->helper_mask, &c->helper_mask) == 0;
  }
  ~HelperSpawnScope() {
    if (active) sched_setaffinity(0, sizeof saved, &saved);
  }
};

// stream-ordered device buffer
template <class T>
struct DBuf {
  T* p = nullptr;
  size_t n = 0;
  Ctx* c = nullptr;
  DBuf() {}
  DBuf(Ctx* ctx, size_t count) { alloc(ctx, count); }
  void alloc(Ctx* ctx, size_t count) {
    release();
    c = ctx;
    n = count;
    if (count) LB_CUDA_CHECK(cudaMallocAsync((void**)&p, count * sizeof(T), ctx->st));
  }
  void release() {
    if (p) cudaFreeAsync(p, c->st);
    p = nullptr;
    n = 0;
  }
  ~DBuf() { release(); }
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  DBuf(DBuf&& o) noexcept : p(o.p), n(o.n), c(o.c) { o.p = nullptr; }
  DBuf& operator=(DBuf&& o) noexcept {
    release();
    p = o.p;
    n = o.n;
    c = o.c;
    o.p = nullptr;
    return *this;
  }
};

struct SpanTimer {
  Ctx* c;
  const char* name;
  std::chrono::steady_clock::time_point t0;
  SpanTimer(Ctx* ctx, const char* n) : c(ctx), name(n) {
    if (c->span_sync) {
      c->sync();
      t0 = std::chrono::steady_clock::now();
    }
  }
  ~SpanTimer() {
    if (c->span_sync) {
      c->sync();
      c->spans[name] += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    }
  }
};

// SparsePolyCommitmentGens<G> (lasso/surge.rs:25-58): one generator stream, three (n, Q, h) views
struct Gens {
  Ctx* ctx = nullptr;
  size_t n_points = 0;
  size_t c = 0, s = 0, num_memories = 0, log_m = 0;
  size_t nv_l = 0, nv_m = 0, nv_d = 0;  // num_vars of the three committed polynomials
  DBuf<fq_t> d_bases_ark;               // n_points x (x, y)
  DBuf<pt_niels> d_table;               // kMsmFullWindows x n_points, T[w][j] = 2^(8w) G_j
  // multiples M[w][j][d-1] = d * T[w][j] (d = 1..128) of the first n_direct generators: the bucket-free MSM of
  // the opening proofs (msm_kernels.cu).  Single-GPU contexts only; empty -> the bucket MSM is used.
  DBuf<pt_niels> d_multiples;
  size_t n_direct = 0;
  // 16-bit multiples M16[j][d-1] = d * G_j (d = 1..32768) of the first n_direct16 generators: the Hyrax row
  // commitments of integer-valued polynomials (3 MB per generator; LASSO_B200_TABLE_GB caps it, default 64)
  DBuf<pt_niels> d_multiples16;
  size_t n_direct16 = 0;
  DBuf<pt_ext> d_centre;  // centring constants 2^15 * sum_{j < R} G_j for R = 2^k, k = 0 .. 31 (entry k; msm_kernels.cu)
};

// DensifiedRepresentation<F, C> (lasso/densified.rs:8-18), device resident
struct Dense {
  Ctx* ctx = nullptr;
  size_t C = 0, s = 0, log_m = 0, m = 0, nv_l = 0, nv_m = 0;
  size_t s_loc = 0, m_loc = 0;  // this rank's share (s / G, m / G): element i' is global element i'*G + rank
  DBuf<uint32_t> d_l_u32;  // (2^nv_l)/G: dim_0..dim_{C-1} | read_0..read_{C-1} | 0..   (dim_usize = first C*s_loc)
  DBuf<uint32_t> d_m_u32;  // (2^nv_m)/G: final_0..final_{C-1} | 0..
  DBuf<fr_t> d_l_fr;       // combined_l_variate_polys (this rank's low-bit shard)
  DBuf<fr_t> d_m_fr;       // combined_log_m_variate_polys
  const uint32_t* nz() const { return d_l_u32.p; }
  const fr_t* dim(size_t i) const { return d_l_fr.p + i * s_loc; }
  const fr_t* read(size_t i) const { return d_l_fr.p + (C + i) * s_loc; }
  const fr_t* fin(size_t i) const { return d_m_fr.p + i * m_loc; }
};

// ark-serialize (compressed) writer
struct ByteWriter {
  std::vector<uint8_t> b;
  void u64(uint64_t v) {
    for (int i = 0; i < 8; i++) b.push_back((uint8_t)(v >> (8 * i)));
  }
  void fr(const fr_t& f) {
    uint8_t t[32];
    fr_to_bytes(f, t);
    b.insert(b.end(), t, t + 32);
  }
  void raw(const void* p, size_t n) { b.insert(b.end(), (const uint8_t*)p, (const uint8_t*)p + n); }
  void vec_fr(const std::vector<fr_t>& v) {
    u64(v.size());
    for (auto& f : v) fr(f);
  }
  void arr_fr(const std::vector<fr_t>& v) {
    for (auto& f : v) fr(f);
  }
  void vec_pts(const std::vector<uint8_t>& comp) {  // comp = 32 B per point
    u64(comp.size() / 32);
    raw(comp.data(), comp.size());
  }
};

inline size_t log2_exact_or_ceil(size_t x) {  // utils/math.rs:27-35 Math::log_2
  if ((x & (x - 1)) == 0) return (size_t)__builtin_ctzll((unsigned long long)x);
  return 64 - (size_t)__builtin_clzll((unsigned long long)x);
}
inline size_t next_pow2(size_t x) {
  size_t p = 1;
  while (p < x) p <<= 1;
  return p;
}

// entry points implemented in prover.cu
int bind_host_threads(int device, cpu_set_t* helper_mask, bool* have_helper_mask);  // -> NUMA node or -1
Ctx* ctx_create(int device);
void ctx_destroy(Ctx*);
Gens* gens_create(Ctx*, const uint64_t* stream_affine, size_t n_points, size_t c, size_t s, size_t num_memories,
                  size_t log_m);
size_t gens_points_needed(size_t c, size_t s, size_t num_memories, size_t log_m);
Dense* densify(Ctx*, const uint64_t* indices, size_t n_lookups, size_t C, size_t log_m, int* err);
// the same on an n x C matrix already on the context's device (dtype: kDzU64 .. kDzI32, element strides)
Dense* densify_device(Ctx*, const void* d_idx, int dtype, size_t n_lookups, size_t C, int64_t row_stride, int64_t col_stride,
                      size_t log_m, cudaStream_t producer, int* err);
std::vector<uint8_t> commit(Ctx*, const Dense&, const Gens&);
std::vector<uint8_t> prove(Ctx*, const Strategy& S, Dense&, const std::vector<fr_t>& r, const Gens&,
                           const std::string& transcript_label, const std::string& tape_label, const fr_t& tape_seed,
                           std::vector<fr_t>* challenges);
void sample_generators(const std::string& label, size_t count, uint64_t* out_affine);

// comm.cu
void comm_unique_id(uint8_t out[128]);
void comm_init(Ctx*, const uint8_t id[128], int rank, int world);
void comm_destroy(Ctx*);
void comm_allgather(Ctx*, const void* d_send, void* d_recv, size_t bytes_per_rank);
// every rank holds the low-bit shard (n_loc elements) of a vector; d_out <- the whole vector (n_loc * G), on every rank
void comm_gather_vector(Ctx*, const fr_t* d_shard, size_t n_loc, fr_t* d_scratch, fr_t* d_out);
// every rank holds one element per polynomial (ptrs[k][0], or base[k*stride] when ptrs == null);
// d_out[k*G + g] <- rank g's element of polynomial k
// `extra` (may be null): one more single-element polynomial, gathered as polynomial number npolys
void comm_gather_heads(Ctx*, fr_t* const* d_ptrs, const fr_t* base, size_t stride, int npolys, const fr_t* extra, fr_t* d_out);
void pack_heads(Ctx*, fr_t* const* d_ptrs, const fr_t* base, size_t stride, int npolys, fr_t* d_out);

}  // namespace lb
