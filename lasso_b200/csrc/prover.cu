// lasso_b200 — the host prover: mirrors the reference's
//   DensifiedRepresentation::from_lookup_indices / commit      (src/lasso/densified.rs:21-96)
//   SparsePolynomialEvaluationProof::prove                      (src/lasso/surge.rs:118-211)
//   MemoryCheckingProof / ProductLayerProof / HashLayerProof    (src/lasso/memory_checking.rs)
//   BatchedGrandProductArgument::prove                          (src/subprotocols/grand_product.rs:100-201)
//   SumcheckInstanceProof::{prove_arbitrary, prove_cubic_batched} (src/subprotocols/sumcheck.rs)
//   PolyEvalProof / DotProductProofLog / BulletReductionProof   (src/poly/dense_mlpoly.rs:301-359,
//                                                                src/subprotocols/{dot_product,bullet}.rs)
// with every field/curve loop on the GPU and only the Fiat–Shamir transcript, the round-polynomial
// interpolation and O(log n)-sized vector glue on the host.  One host<->device round trip per sumcheck
// round ((deg+1) x 32 B down, the challenge travels as a kernel argument).
//
// Bulletproofs on a GPU (bullet.rs:73-142): the reference folds the generator vector every round,
// G_L[i] <- u^-1 G_L[i] + u G_R[i] — 2n serial variable-base scalar multiplications per opening.  Here the
// generators are never folded: round k's L and R are MSMs over the ORIGINAL generators with scalars
// a[i] * W_k[t] (W_k = the 2^k products of u_r^{+-1}), so every group operation of the proof is a row-MSM
// over one fixed table T[w][j] = 2^(8w) G_j.  The group elements are identical; only the schedule differs.
#include "prover.cuh"

#include <sched.h>

#include <cctype>
#include <mutex>
#include <thread>

#include "host_fq64.hpp"

namespace lb {

std::atomic<unsigned long long> g_launches{0};

// ---------------------------------------------------------------------------------------------- context
__global__ void publish_kernel(const uint32_t* src, int nwords, uint32_t* mapped, uint32_t seq) {
  for (int i = threadIdx.x; i < nwords; i += blockDim.x) mapped[i] = src[i];
  __threadfence_system();
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    *((volatile uint32_t*)(mapped + 1024)) = seq;
  }
}
void Ctx::d2h_small(void* dst, const void* src, size_t bytes) {
  const uint32_t seq = ++mapped_seq;
  publish_kernel<<<1, 128, 0, st>>>((const uint32_t*)src, (int)((bytes + 3) / 4), d_mapped, seq);
  g_launches += 1;
  wait_flag(seq);
  memcpy(dst, (const void*)h_mapped, bytes);
}
// One element = five 64-bit words, each carrying 51 value bits and the 13-bit tag of its message (common.cuh): a
// word is accepted only when it shows the tag, so neither the order in which the device's stores become visible
// nor the width of the store instruction matters.  Consumed slots are zeroed.
void Ctx::pub_wait_raw(const PubDst& p, int writer, int count, uint32_t* out) {
  if (!h_pub || !p.ndst) throw std::runtime_error("no publication buffer for this message");
  if ((size_t)count > (size_t)kPubElems) throw std::runtime_error("message larger than a publication region");
  volatile unsigned long long* base = h_pub + ((size_t)writer * kPubRegions + p.region) * kPubElems * kPubSlotWords;
  const uint32_t tag = p.tag;
  auto t0 = std::chrono::steady_clock::now();
  unsigned spins = 0;
  for (int v = 0; v < count; v++) {
    volatile unsigned long long* s = base + (size_t)v * kPubSlotWords;
    unsigned long long w[5];
    for (int k = 0; k < 5; k++) {
      while (pub_tag_of(w[k] = s[k]) != tag) {
        __builtin_ia32_pause();
        if ((++spins & 0xffff) == 0) {  // surface kernel faults instead of spinning forever
          double dt = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
          if (dt > 0.5) LB_CUDA_CHECK(cudaStreamQuery(st) == cudaErrorNotReady ? cudaSuccess : cudaStreamSynchronize(st));
          if (dt > 120.0) throw std::runtime_error("timeout waiting for a device result");
        }
      }
      w[k] &= kPubValueMask;
    }
    for (int k = 0; k < 5; k++) s[k] = 0;  // consumed
    pub_decode(w, out + 8 * (size_t)v);
  }
}
void Ctx::fin_wait(const Finalize& f, fr_t* dst, int count) {
  if (!f.pub.all) {
    pub_wait_raw(f.pub, rank, count, (uint32_t*)dst);
    return;
  }
  // one proof sharded over `world` GPUs: every rank stored its partial sums here; add the residues (mod l)
  std::vector<fr_t> tmp((size_t)count);
  for (int w = 0; w < world; w++) {
    pub_wait_raw(f.pub, w, count, (uint32_t*)(w == 0 ? dst : tmp.data()));
    if (w)
      for (int v = 0; v < count; v++) dst[v] = fr_add(dst[v], tmp[v]);
  }
}
void Ctx::wait_points(const PubDst& p, int npoints, uint32_t* xyz) { pub_wait_raw(p, rank, 3 * npoints, xyz); }
void Ctx::wait_flag(uint32_t seq) {
  volatile uint32_t* flag = h_mapped + 1024;
  auto t0 = std::chrono::steady_clock::now();
  unsigned spins = 0;
  while (*flag != seq) {
    __builtin_ia32_pause();
    if ((++spins & 0xffff) == 0) {  // surface kernel faults instead of spinning forever
      if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 0.5) {
        LB_CUDA_CHECK(cudaStreamQuery(st) == cudaErrorNotReady ? cudaSuccess : cudaStreamSynchronize(st));
        if (std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count() > 120.0)
          throw std::runtime_error("timeout waiting for a device result");
      }
    }
  }
  __sync_synchronize();
}
// ---- host-thread placement (one process per GPU on a multi-socket node) -------------------------------------------
// The prover's host side is ONE latency-critical thread (it spins on the round messages and hashes them) plus short
// bursts of helper threads (staging the index matrix).  bind_host_threads pins the CALLING thread to one dedicated
// physical core of the NUMA node its GPU hangs off — a different core for every GPU of the node, spread over the
// node's cores — and gives the helper threads the rest of the node (all its CPUs minus the dedicated cores and their
// SMT siblings).  A spinning thread that shares a core with anything else loses milliseconds per proof.
static std::vector<int> parse_cpulist(const std::string& path) {
  std::vector<int> out;
  FILE* f = fopen(path.c_str(), "r");
  if (!f) return out;
  char buf[4096] = {0};
  if (fgets(buf, sizeof buf, f)) {
    for (char* tok = strtok(buf, ",\n"); tok; tok = strtok(nullptr, ",\n")) {  // "0-31,64-95"
      int lo = 0, hi = 0;
      if (sscanf(tok, "%d-%d", &lo, &hi) == 2) {
      } else if (sscanf(tok, "%d", &lo) == 1) {
        hi = lo;
      } else {
        continue;
      }
      for (int cpu = lo; cpu <= hi; cpu++) out.push_back(cpu);
    }
  }
  fclose(f);
  return out;
}
static int numa_node_of_device(int device) {
  char busid[64] = {0};
  if (cudaDeviceGetPCIBusId(busid, sizeof busid, device) != cudaSuccess) return -1;
  for (char* p = busid; *p; p++) *p = (char)tolower(*p);
  int node = -1;
  FILE* f = fopen((std::string("/sys/bus/pci/devices/") + busid + "/numa_node").c_str(), "r");
  if (!f) return -1;
  if (fscanf(f, "%d", &node) != 1) node = -1;
  fclose(f);
  return node;
}
// -> NUMA node or -1.  helper_mask (may be null) receives the CPUs for helper threads.
int bind_host_threads(int device, cpu_set_t* helper_mask, bool* have_helper_mask) {
  try {
    if (have_helper_mask) *have_helper_mask = false;
    const int node = numa_node_of_device(device);
    if (node < 0) return -1;
    const std::vector<int> cpus = parse_cpulist("/sys/devices/system/node/node" + std::to_string(node) + "/cpulist");
    if (cpus.empty()) return -1;
    // GPUs on this node, and this GPU's index among them
    int ndev = 0, cnt = 0, idx = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess) ndev = device + 1;
    for (int d = 0; d < ndev; d++)
      if (numa_node_of_device(d) == node) {
        if (d < device) idx++;
        cnt++;
      }
    if (cnt < 1) cnt = 1;
    // physical cores = CPUs that are the first of their sibling list
    std::vector<int> phys;
    std::map<int, std::vector<int>> sib;
    for (int cpu : cpus) {
      std::vector<int> s = parse_cpulist("/sys/devices/system/cpu/cpu" + std::to_string(cpu) + "/topology/thread_siblings_list");
      if (s.empty()) s.push_back(cpu);
      sib[cpu] = s;
      if (s[0] == cpu) phys.push_back(cpu);
    }
    if (phys.empty()) phys = cpus;
    auto dedicated = [&](int k) { return phys[(size_t)(k + 1) * phys.size() / (size_t)(cnt + 1) % phys.size()]; };
    cpu_set_t helpers;
    CPU_ZERO(&helpers);
    for (int cpu : cpus)
      if (cpu < CPU_SETSIZE) CPU_SET(cpu, &helpers);
    for (int k = 0; k < cnt; k++)
      for (int c2 : sib[dedicated(k)])
        if (c2 < CPU_SETSIZE) CPU_CLR(c2, &helpers);
    if (CPU_COUNT(&helpers) == 0)
      for (int cpu : cpus)
        if (cpu < CPU_SETSIZE) CPU_SET(cpu, &helpers);
    cpu_set_t mine;
    CPU_ZERO(&mine);
    const int my_cpu = dedicated(idx);
    if (my_cpu >= CPU_SETSIZE) return -1;
    CPU_SET(my_cpu, &mine);
    if (sched_setaffinity(0, sizeof mine, &mine) != 0) return -1;
    if (helper_mask && have_helper_mask) {
      *helper_mask = helpers;
      *have_helper_mask = true;
    }
    return node;
  } catch (...) {
    return -1;
  }
}
Ctx* ctx_create(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    throw std::runtime_error("lasso_b200 needs a CUDA device (sm_100a); there is no CPU fallback");
  if (device < 0 || device >= count) throw std::runtime_error("invalid device id");
  LB_CUDA_CHECK(cudaSetDevice(device));
  {
  }
  std::unique_ptr<Ctx> c(new Ctx());
  c->device = device;
  {
    const char* nb = getenv("LASSO_B200_NUMA_BIND");
    if (nb && nb[0] == '1') bind_host_threads(device, &c->helper_mask, &c->have_helper_mask);
  }
  LB_CUDA_CHECK(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
  cudaMemPool_t pool;
  LB_CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, device));
  uint64_t thr = UINT64_MAX;
  LB_CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
  c->h_pin_bytes = 8u << 20;
  LB_CUDA_CHECK(cudaMallocHost((void**)&c->h_pin, c->h_pin_bytes));
  c->partial_elems = (size_t)bound_max_chunks() * 16384 + 65536;
  LB_CUDA_CHECK(cudaMalloc((void**)&c->d_partial, c->partial_elems * sizeof(fr_t)));
  c->small_elems = 65536;
  LB_CUDA_CHECK(cudaMalloc((void**)&c->d_small, c->small_elems * sizeof(fr_t)));
  LB_CUDA_CHECK(cudaMalloc((void**)&c->d_eq_scratch, (size_t)(4096 + (1 << 17) + 4096) * sizeof(fr_t)));
  LB_CUDA_CHECK(cudaMalloc((void**)&c->d_flag, 64));
  LB_CUDA_CHECK(cudaMemset(c->d_flag, 0, 64));
  {
    const char* nm = getenv("LASSO_B200_NO_MAPPED");
    if (!(nm && nm[0] == '1')) {
      LB_CUDA_CHECK(cudaHostAlloc((void**)&c->h_mapped, Ctx::kMappedBytes, cudaHostAllocMapped));
      memset(c->h_mapped, 0, Ctx::kMappedBytes);
      LB_CUDA_CHECK(cudaHostGetDevicePointer((void**)&c->d_mapped, c->h_mapped, 0));
      LB_CUDA_CHECK(cudaHostAlloc((void**)&c->h_pub, Ctx::kPubBytes, cudaHostAllocMapped));
      memset(c->h_pub, 0, Ctx::kPubBytes);
      c->h_pub_owned = true;
      LB_CUDA_CHECK(cudaHostGetDevicePointer((void**)&c->d_pub_reader[0], c->h_pub, 0));
    }
  }
  msm_init_device();      // per-device function attributes (dynamic shared memory opt-in)
  msm_large_init_device();
  densify_init_device();
  LB_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_aux, cudaEventDisableTiming));
  LB_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_stage, cudaEventDisableTiming));
  LB_CUDA_CHECK(cudaEventCreateWithFlags(&c->ev_input, cudaEventDisableTiming));
  const char* sp = getenv("LASSO_B200_SPANS");
  c->span_sync = sp && sp[0] == '1';
  return c.release();
}
void ctx_destroy(Ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->st);
  cudaFree(c->d_partial);
  cudaFree(c->d_small);
  cudaFree(c->d_eq_scratch);
  cudaFree(c->d_flag);
  if (c->ev_aux) cudaEventDestroy(c->ev_aux);
  if (c->ev_stage) cudaEventDestroy(c->ev_stage);
  if (c->ev_input) cudaEventDestroy(c->ev_input);
  if (c->h_stage) cudaFreeHost(c->h_stage);
  if (c->h_mapped) cudaFreeHost(c->h_mapped);
  if (c->h_pub && c->h_pub_owned) cudaFreeHost(c->h_pub);
  cudaFreeHost(c->h_pin);
  cudaStreamDestroy(c->st);
  delete c;
}

static FrVec to_frvec(const std::vector<fr_t>& v, size_t off, size_t n) {
  if (n > 32) throw std::runtime_error("challenge vector too long");
  FrVec f;
  for (size_t i = 0; i < n; i++) f.v[i] = v[off + i];
  return f;
}
// eq(r) table on the device (eq_poly.rs:21-38)
static void eq_evals_dev(Ctx* c, const std::vector<fr_t>& r, size_t off, size_t ell, fr_t* out) {
  launch_eq_evals(to_frvec(r, off, ell), (int)ell, out, c->d_eq_scratch, c->st);
  g_launches += ell <= 11 ? 1 : (ell <= 22 ? 3 : 5);
}

// ---------------------------------------------------------------------------------------------- generators
size_t gens_points_needed(size_t c, size_t s, size_t num_memories, size_t log_m) {
  size_t nv_l = log2_exact_or_ceil(next_pow2(2 * c * s));
  size_t nv_m = log2_exact_or_ceil(next_pow2(c)) + log_m;
  size_t nv_d = log2_exact_or_ceil(next_pow2(num_memories * s));
  size_t mx = std::max(nv_l, std::max(nv_m, nv_d));
  return ((size_t)1 << (mx - mx / 2)) + 2;
}
Gens* gens_create(Ctx* c, const uint64_t* stream_affine, size_t n_points, size_t cc, size_t s, size_t num_memories,
                  size_t log_m) {
  if (n_points < gens_points_needed(cc, s, num_memories, log_m)) return nullptr;
  std::unique_ptr<Gens> g(new Gens());
  g->ctx = c;
  g->n_points = n_points;
  g->c = cc;
  g->s = s;
  g->num_memories = num_memories;
  g->log_m = log_m;
  g->nv_l = log2_exact_or_ceil(next_pow2(2 * cc * s));
  g->nv_m = log2_exact_or_ceil(next_pow2(cc)) + log_m;
  g->nv_d = log2_exact_or_ceil(next_pow2(num_memories * s));
  g->d_bases_ark.alloc(c, n_points * 2);
  LB_CUDA_CHECK(cudaMemcpyAsync(g->d_bases_ark.p, stream_affine, n_points * 64, cudaMemcpyHostToDevice, c->st));
  g->d_table.alloc(c, (size_t)kMsmFullWindows * n_points);
  launch_build_table(g->d_bases_ark.p, n_points, g->d_table.p, n_points, kMsmFullWindows, c->st);
  g_launches += kMsmFullWindows;
  {
    // widest opening: R_size = 2^(nv - nv/2) generators + Q + h (dense_mlpoly.rs:301-316)
    size_t nv = std::max(g->nv_l, std::max(g->nv_m, g->nv_d));
    size_t nd = ((size_t)1 << (nv - nv / 2)) + 2;
    const char* off = getenv("LASSO_B200_NO_MULTIPLES");
    // The tables are an optimisation: if the device cannot hold them (cap, or an allocation failure on a smaller
    // or busier GPU) the prover silently keeps the bucket / 8-bit paths — outputs do not depend on it.
    // One proof sharded over G GPUs: the openings run replicated (every rank needs the 8-bit multiples of all
    // nd generators), the Hyrax commitments are column-sharded (a rank needs the 16-bit multiples of ITS columns
    // only: 1/G of the table per GPU).
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const size_t G = (size_t)c->world, gr = (size_t)c->rank;
    const size_t bytes8 = (size_t)kMsmFullWindows * nd * 128 * sizeof(pt_niels);
    if (nd <= n_points && !(off && off[0] == '1') && bytes8 < free_b / 2) {
      g->n_direct = nd;
      g->d_multiples.alloc(c, (size_t)kMsmFullWindows * nd * 128);
      launch_build_multiples(g->d_table.p, n_points, nd, kMsmFullWindows, g->d_multiples.p, c->st);
      g_launches += 1;
      const char* cap = getenv("LASSO_B200_TABLE_GB");
      const double cap_gb = cap ? atof(cap) : 64.0;
      const size_t ncols16 = (nd - 2) / G;  // this rank's columns: generators j * G + rank
      const size_t bytes16 = ncols16 * 32768 * sizeof(pt_niels);
      if (ncols16 >= 1 && (nd - 2) % G == 0 && (double)bytes16 <= cap_gb * 1e9 && bytes16 < (free_b - bytes8) / 2) {
        g->n_direct16 = ncols16;
        g->d_multiples16.alloc(c, ncols16 * 32768);
        launch_build_multiples16(g->d_table.p, g->d_multiples.p, nd, ncols16, G, gr, g->d_multiples16.p, c->st);
        g_launches += 1;
        g->d_centre.alloc(c, 32);
        for (size_t k = 0; ((size_t)1 << k) <= ncols16 && k < 32; k++) {  // one constant per power-of-two (local) row length
          launch_centre_constant(g->d_multiples16.p, 1 << k, g->d_centre.p + k, c->st);
          g_launches += 1;
        }
      }
    }
  }
  c->sync();
  return g.release();
}

// ---------------------------------------------------------------------------------------------- sharding helpers
// One proof sharded over G = c->world GPUs: every array of global length n >= G is partitioned by the low
// log2(G) index bits (rank g holds X[i*G + g]); see comm.cu.  With G == 1 all of this is the identity.
static inline size_t loc(const Ctx* c, size_t n) {
  if (n % (size_t)c->world) throw std::runtime_error("array shorter than the number of GPUs");
  return n / (size_t)c->world;
}
// a few field elements computed on the device -> host, summed over the ranks of a sharded proof: one tiny kernel
// publishes them as a tagged message to every process (common.cuh PubDst)
__global__ void publish_fr_kernel(const fr_t* src, int count, PubDst pub) {
  for (int v = threadIdx.x; v < count; v += blockDim.x) {
    const fr_t x = src[v];
    pub_store(pub, v, x.v);
  }
}
// In two halves so that host work can sit between the launch and the wait; `f.pub.ndst == 0` after _begin: no
// publication buffers, _end copies synchronously.
static Finalize reduce_to_host_begin(Ctx* c, fr_t* d_buf, int count) {
  if (!c->h_pub || count > kPubElems) {
    if (c->world > 1) throw std::runtime_error("sharded proof without publication buffers");
    Finalize f{};
    f.pub.ndst = 0;
    return f;
  }
  Finalize f = c->fin_begin(true);
  publish_fr_kernel<<<1, 128, 0, c->st>>>(d_buf, count, f.pub);
  LB_LAUNCH_CHECK();
  g_launches += 1;
  return f;
}
static void reduce_to_host_end(Ctx* c, const Finalize& f, fr_t* d_buf, int count, fr_t* h_out) {
  if (f.pub.ndst == 0) {
    c->d2h(h_out, d_buf, (size_t)count * sizeof(fr_t));
    return;
  }
  c->fin_wait(f, h_out, count);
}
static void reduce_to_host(Ctx* c, fr_t* d_buf, int count, fr_t* h_out) {
  const Finalize f = reduce_to_host_begin(c, d_buf, count);
  reduce_to_host_end(c, f, d_buf, count, h_out);
}
// this rank's shard of eq(r[off .. off+ell)) (eq_poly.rs:21-38): eq[i*G + g] = eq_hi[i] * eq_lo[g] where
// eq_lo is the table of the LAST log2(G) coordinates (they bind the low index bits: r[0] <-> MSB)
static void eq_evals_shard(Ctx* c, const std::vector<fr_t>& r, size_t off, size_t ell, fr_t* out) {
  const size_t lg = (size_t)c->lg_world;
  if (ell < lg) throw std::runtime_error("eq table smaller than the number of GPUs");
  eq_evals_dev(c, r, off, ell - lg, out);
  if (lg == 0) return;
  fr_t k = fr_one();
  for (size_t j = 0; j < lg; j++) {
    const fr_t& rj = r[off + ell - lg + j];
    bool bit = (c->rank >> (lg - 1 - j)) & 1;
    k = fr_mul(k, bit ? rj : fr_sub(fr_one(), rj));
  }
  launch_scale(out, out, (size_t)1 << (ell - lg), k, c->st);
  g_launches += 1;
}

// ---------------------------------------------------------------------------------------------- MSM helpers
// Row-MSMs over the generator table with the bucket kernels.  Column-sharded (replicated == false, G > 1): `d_scal`
// holds this rank's columns (ncols per row, local column c' = generator c'*G + rank), the per-row partial points
// of every rank are all-gathered and added ("bucket-sum reduce" = gather-then-add).  Replicated: every rank
// passes the same full rows and computes the same points, no exchange.  Returns nrows compressed points.
static std::vector<uint8_t> msm_rows(Ctx* c, const Gens& g, const void* d_scal, int limbs, size_t row_stride, int nrows,
                                     int ncols, int nw, bool replicated) {
  const int G = replicated ? 1 : c->world, gr = replicated ? 0 : c->rank;
  std::vector<uint8_t> out((size_t)nrows * 32);
  const bool few = nrows <= 8;
  DBuf<pt_ext> part(c, msm_partials_count(nrows, ncols, nw));
  if (G == 1 && !few) {  // the common single-GPU commit: normalise on the device
    DBuf<uint32_t> comp(c, (size_t)nrows * 8);
    launch_msm_rows(g.d_table.p, g.n_points, 1, d_scal, limbs, row_stride, nrows, ncols, nw, 1, 0, part.p, nullptr, comp.p,
                    nullptr, c->st);
    g_launches += 2;
    c->d2h(out.data(), comp.p, out.size());
    return out;
  }
  // raw partial points -> (gather over ranks) -> sum -> normalise
  DBuf<uint32_t> raw(c, (size_t)(G + 1) * nrows * 32);
  uint32_t* mine = raw.p + (size_t)G * nrows * 32;  // scratch slot for this rank's partials
  launch_msm_rows(g.d_table.p, g.n_points, 1, d_scal, limbs, row_stride, nrows, ncols, nw, G, gr, part.p, nullptr, nullptr,
                  G == 1 ? raw.p : mine, c->st);
  g_launches += 2;
  if (G > 1) comm_allgather(c, mine, raw.p, (size_t)nrows * 128);
  if (few) {
    uint32_t xyzt[8 * 32];
    if (G > 1) {
      launch_sum_raw_points(raw.p, G, nrows, mine, nullptr, nullptr, c->st);
      g_launches += 1;
      c->d2h(xyzt, mine, (size_t)nrows * 128);
    } else {
      c->d2h(xyzt, raw.p, (size_t)nrows * 128);
    }
    // a couple of points per Bulletproofs round: invert on the host (3 us vs ~100 us on one GPU thread)
    for (int i = 0; i < nrows; i++) h64::compress_xyz(xyzt + 32 * i, out.data() + 32 * i);
    return out;
  }
  DBuf<uint32_t> comp(c, (size_t)nrows * 8);
  launch_sum_raw_points(raw.p, G, nrows, nullptr, comp.p, nullptr, c->st);
  g_launches += 1;
  c->d2h(out.data(), comp.p, out.size());
  return out;
}
// replicated rows of Montgomery Fr scalars over the generators [0, ncols) (the openings when the multiples tables
// are not available): every rank computes the same points
static std::vector<uint8_t> msm_rows_fr(Ctx* c, const Gens& g, const fr_t* d_scal_mont, int nrows, int ncols) {
  DBuf<fr_t> canon(c, (size_t)nrows * ncols);
  launch_canonicalize(d_scal_mont, canon.p, (size_t)nrows * ncols, c->d_flag, c->st);
  g_launches += 1;
  return msm_rows(c, g, canon.p, 8, (size_t)ncols, nrows, ncols, kMsmFullWindows, true);
}

// DensePolynomial::commit (dense_mlpoly.rs:152-181) for an integer-valued polynomial of 2^nv entries viewed as
// L x R; this rank holds, for every row, the R/G columns congruent to its rank (= its low-bit shard of the array)
static std::vector<uint8_t> commit_u32(Ctx* c, const Gens& g, const uint32_t* d_vals_loc, size_t nv, unsigned max_bits) {
  size_t L = (size_t)1 << (nv / 2), R = (size_t)1 << (nv - nv / 2);
  if (R + 2 > g.n_points) throw std::runtime_error("generator stream too short for this polynomial");
  int nw = msm_windows_for_bits(max_bits);
  if (nw > 5) throw std::runtime_error("u32 MSM path: scalars wider than 32 bits");
  const int G = c->world;
  size_t R_loc = loc(c, R);
  if (g.d_multiples.p && R + 2 <= g.n_direct && L > 8) {
    // rows as direct sums over the digit-multiples tables (msm_kernels.cu): one table entry per committed integer
    std::vector<uint8_t> out(L * 32);
    DBuf<pt_ext> part(c, L);
    DBuf<uint32_t> comp(c, L * 8);
    const bool wide = R_loc <= g.n_direct16;
    size_t lg_rloc = 0;
    while (((size_t)1 << lg_rloc) < R_loc) lg_rloc++;
    const pt_niels* m16 = wide ? g.d_multiples16.p : nullptr;
    const pt_ext* k16 = wide ? g.d_centre.p + lg_rloc : nullptr;
    if (G == 1) {  // normalised on the device
      launch_msm_rows_direct_u32(g.d_multiples.p, g.n_direct, m16, k16, d_vals_loc, R, (int)L, (int)R, nw, 1, 0, part.p, nullptr,
                                 comp.p, nullptr, c->st);
      g_launches += 2;
    } else {  // this rank's columns of every row -> partial points -> gather-then-add over the ranks
      DBuf<uint32_t> raw(c, (size_t)(G + 1) * L * 32);
      uint32_t* mine = raw.p + (size_t)G * L * 32;
      launch_msm_rows_direct_u32(g.d_multiples.p, g.n_direct, m16, k16, d_vals_loc, R_loc, (int)L, (int)R_loc, nw, G, c->rank,
                                 part.p, nullptr, nullptr, mine, c->st);
      comm_allgather(c, mine, raw.p, L * 128);
      launch_sum_raw_points(raw.p, G, (int)L, nullptr, comp.p, nullptr, c->st);
      g_launches += 3;
      c->d2h(out.data(), comp.p, out.size());
      return out;
    }
    c->d2h(out.data(), comp.p, out.size());
    return out;
  }
  return msm_rows(c, g, d_vals_loc, 1, R_loc, (int)L, (int)R_loc, nw, false);
}

// ---------------------------------------------------------------------------------------------- densify
// The shape checks both densify entry points share and the header of their result (nullptr with *err = 4 if invalid).
static std::unique_ptr<Dense> dense_header(Ctx* c, size_t n, size_t C, size_t log_m, int* err) {
  *err = 0;
  if (n == 0 || C == 0 || C > 16 || log_m < 1 || log_m > 28) {
    *err = 4;
    return nullptr;
  }
  const size_t G = (size_t)c->world;
  std::unique_ptr<Dense> d(new Dense());
  d->ctx = c;
  d->C = C;
  d->s = next_pow2(n);
  d->log_m = log_m;
  d->m = (size_t)1 << log_m;
  d->nv_l = log2_exact_or_ceil(next_pow2(2 * C * d->s));
  d->nv_m = log2_exact_or_ceil(next_pow2(C)) + log_m;
  if (G > 1 && (d->s < 2 * G || d->m < 2 * G)) {
    *err = 4;
    return nullptr;
  }
  d->s_loc = d->s / G;
  d->m_loc = d->m / G;
  return d;
}

// The device half both entry points share once the index matrix is on the device: the four arrays of d and their zero
// padding, the stable sort by address (densify_kernels.cu) and DensePolynomial::from_usize + merge.  Queued on the
// context stream, no sync.
static void densify_on_device(Ctx* c, Dense* d, const DzSource& src, size_t n) {
  const size_t G = (size_t)c->world, gr = (size_t)c->rank, C = d->C, s = d->s, s_loc = d->s_loc, m_loc = d->m_loc;
  const size_t nl = ((size_t)1 << d->nv_l) / G, nm = ((size_t)1 << d->nv_m) / G;  // local lengths
  d->d_l_u32.alloc(c, nl);
  d->d_m_u32.alloc(c, nm);
  d->d_l_fr.alloc(c, nl);
  d->d_m_fr.alloc(c, nm);
  DBuf<uint32_t> scratch(c, densify_scratch_words(s, (int)C, d->log_m));
  if (nl > 2 * C * s_loc) LB_CUDA_CHECK(cudaMemsetAsync(d->d_l_u32.p + 2 * C * s_loc, 0, (nl - 2 * C * s_loc) * 4, c->st));
  if (nm > C * m_loc) LB_CUDA_CHECK(cudaMemsetAsync(d->d_m_u32.p + C * m_loc, 0, (nm - C * m_loc) * 4, c->st));
  g_launches += launch_densify(src, n, s, (int)C, d->log_m, (int)G, (int)gr, scratch.p, d->d_l_u32.p, s_loc,
                               d->d_l_u32.p + C * s_loc, s_loc, d->d_m_u32.p, m_loc, c->st);
  launch_from_u32(d->d_l_u32.p, d->d_l_fr.p, nl, c->st);  // DensePolynomial::from_usize + merge
  launch_from_u32(d->d_m_u32.p, d->d_m_fr.p, nm, c->st);
  g_launches += 2;
}

Dense* densify(Ctx* c, const uint64_t* indices, size_t n, size_t C, size_t log_m, int* err) {
  SpanTimer sp(c, "Densify");
  std::unique_ptr<Dense> d = dense_header(c, n, C, log_m, err);
  if (!d) return nullptr;
  const size_t G = (size_t)c->world, gr = (size_t)c->rank;
  const size_t s = d->s, m = d->m, s_loc = d->s_loc, m_loc = d->m_loc;
  const size_t nl = ((size_t)1 << d->nv_l) / G, nm = ((size_t)1 << d->nv_m) / G;  // local lengths
  {
    const char* hd = getenv("LASSO_B200_HOST_DENSIFY");
    const char* gd = getenv("LASSO_B200_GPU_DENSIFY");
    // The device path (a stable radix sort by address, densify_kernels.cu) replaces the C host threads of the
    // sequential scan: ~0.5 ms of kernels instead of ~3 ms of host time at 2^20 lookups, and nothing that slows
    // down when several processes share the host (one process per GPU).  Tiny inputs stay on the host (the ~20
    // launches cost more than the scan).
    const bool want_gpu = (gd && gd[0] == '1') || s >= ((size_t)1 << 15) || G > 1;
    if (densify_gpu_supported(s, log_m) && want_gpu && !(hd && hd[0] == '1')) {
      // upload the raw index matrix, derive dim / read / final on the device.  When one proof is sharded every rank
      // does this for the whole sequence and stores only its shard.
      // narrow usize -> u32 (and range-check, densified.rs:46) while staging into pinned memory: half the PCIe
      // bytes and a full-rate copy.  Pipelined: the matrix is cut into pieces, a few host threads narrow them
      // round-robin, and the upload of a piece starts as soon as it is staged (the copy of the early pieces overlaps
      // the narrowing of the later ones).
      if (c->stage_busy) {  // the previous call's upload may still be reading the staging buffer
        LB_CUDA_CHECK(cudaEventSynchronize(c->ev_stage));
        c->stage_busy = false;
      }
      // One proof sharded over G ranks: every rank stages and uploads only ITS block of rows (1/G of the host work
      // and of the PCIe bytes), the narrowed blocks are all-gathered over NVLink, and every rank sorts the whole
      // sequence on its device and keeps its shard.
      const size_t rows_per = G > 1 ? (((n + G - 1) / G + 3) & ~(size_t)3) : n;  // x C x 4 B: a multiple of 16 bytes
      const size_t row0 = std::min(n, gr * rows_per), row1 = std::min(n, row0 + rows_per);
      const size_t total = (row1 - row0) * C;  // elements this rank stages
      const uint64_t* src = indices + row0 * C;
      uint32_t* stage = c->stage(std::max<size_t>(total, 1));
      DBuf<uint32_t> d_idx(c, G * rows_per * C), d_mine(c, G > 1 ? rows_per * C : 0);
      uint32_t* d_dst = G > 1 ? d_mine.p : d_idx.p;
      {
        const size_t npieces = total >= (1u << 20) ? 64 : 1, nthreads = npieces > 1 ? (total >= (1u << 25) ? 16 : total >= (1u << 22) ? 8 : 4) : 1;
        std::vector<std::atomic<int>> done(npieces);
        for (auto& f : done) f.store(0);
        std::atomic<int> bad{0};
        auto conv = [&](size_t t) {
          if (nthreads > 1) c->helper_thread_enter();
          for (size_t p = t; p < npieces; p += nthreads) {
            const size_t lo = total * p / npieces, hi = total * (p + 1) / npieces;
            int b = 0;
            for (size_t k = lo; k < hi; k++) {
              uint64_t a = src[k];
              if (a >= m) {
                b = 1;
                a = 0;
              }
              stage[k] = (uint32_t)a;
            }
            if (b) bad.store(1);
            done[p].store(1, std::memory_order_release);
          }
        };
        std::vector<std::thread> th;
        std::thread t0;
        {
          HelperSpawnScope spawn(c, nthreads > 1);  // a pinned caller must not hand its single CPU down to the helpers
          for (size_t t = 1; t < nthreads; t++) th.emplace_back(conv, t);
          if (nthreads > 1) t0 = std::thread(conv, 0);
        }
        if (nthreads == 1) conv(0);
        if (G > 1 && total < rows_per * C)  // a short (or empty) last block: the gathered matrix must not carry garbage
          LB_CUDA_CHECK(cudaMemsetAsync(d_mine.p + total, 0, (rows_per * C - total) * sizeof(uint32_t), c->st));
        for (size_t p = 0; p < npieces; p++) {  // this thread feeds the copy engine in order
          while (!done[p].load(std::memory_order_acquire)) __builtin_ia32_pause();
          const size_t lo = total * p / npieces, hi = total * (p + 1) / npieces;
          if (hi > lo)
            LB_CUDA_CHECK(cudaMemcpyAsync(d_dst + lo, stage + lo, (hi - lo) * sizeof(uint32_t), cudaMemcpyHostToDevice, c->st));
        }
        if (t0.joinable()) t0.join();
        for (auto& t : th) t.join();
        LB_CUDA_CHECK(cudaEventRecord(c->ev_stage, c->st));
        c->stage_busy = true;
        bool any_bad = bad.load() != 0;
        if (G > 1) {
          // every rank must reach the same verdict (densified.rs:46): the flags are summed through the round-message path
          fr_t flag = fr_zero(), sum;
          flag.v[0] = any_bad ? 1u : 0u;
          c->h2d(c->d_small, &flag, sizeof flag);
          reduce_to_host(c, c->d_small, 1, &sum);
          any_bad = !fr_is_zero(sum);
        }
        if (any_bad) {
          c->sync();
          *err = 3;
          return nullptr;
        }
        if (G > 1) comm_allgather(c, d_mine.p, d_idx.p, rows_per * C * sizeof(uint32_t));
      }
      DzSource staged;  // n x C u32 row-major, range-checked above
      staged.p = d_idx.p;
      staged.type = kDzU32;
      staged.row_stride = (int64_t)C;
      staged.col_stride = 1;
      densify_on_device(c, d.get(), staged, n);
      // no stream sync here: everything downstream is stream-ordered, and the staging buffer is guarded by ev_stage
      return d.release();
    }
  }
  // host path (memories larger than 2^16 cells): pinned staging, reused across calls: no per-call page faults, and the upload runs at full PCIe rate
  if (c->stage_busy) {
    LB_CUDA_CHECK(cudaEventSynchronize(c->ev_stage));
    c->stage_busy = false;
  }
  uint32_t* l_host = c->stage(nl + nm + (G > 1 ? (2 * s + m) * C : 0));
  uint32_t* m_host = l_host + nl;
  uint32_t* full = m_host + nm;  // G > 1: whole-sequence scratch (every rank runs the full scan, keeps its shard)
  if (nl > 2 * C * s_loc) memset(l_host + 2 * C * s_loc, 0, (nl - 2 * C * s_loc) * sizeof(uint32_t));
  if (nm > C * m_loc) memset(m_host + C * m_loc, 0, (nm - C * m_loc) * sizeof(uint32_t));
  // densified.rs:33-56: per dimension, pad with address 0 and run the (inherently sequential) timestamp
  // counters; dimensions are independent, so one host thread each.
  std::vector<int> bad(C, 0);
  auto work = [&](size_t i) {
    if (i > 0) c->helper_thread_enter();
    uint32_t* dim = G == 1 ? l_host + i * s : full + i * (2 * s + m);
    uint32_t* rd = G == 1 ? l_host + (C + i) * s : dim + s;
    uint32_t* fin = G == 1 ? m_host + i * m : dim + 2 * s;
    memset(fin, 0, m * sizeof(uint32_t));
    for (size_t k = 0; k < s; k++) {
      uint64_t addr = k < n ? indices[k * C + i] : 0;
      if (addr >= m) {
        bad[i] = 1;
        return;
      }
      dim[k] = (uint32_t)addr;
      uint32_t ts = fin[addr];
      rd[k] = ts;
      fin[addr] = ts + 1;
    }
    if (G > 1) {  // keep the low-bit shard
      uint32_t* ld = l_host + i * s_loc;
      uint32_t* lr = l_host + (C + i) * s_loc;
      uint32_t* lf = m_host + i * m_loc;
      for (size_t k = 0; k < s_loc; k++) {
        ld[k] = dim[k * G + gr];
        lr[k] = rd[k * G + gr];
      }
      for (size_t k = 0; k < m_loc; k++) lf[k] = fin[k * G + gr];
    }
  };
  {
    std::vector<std::thread> th;
    {
      HelperSpawnScope spawn(c, C > 1);
      for (size_t i = 1; i < C; i++) th.emplace_back(work, i);
    }
    work(0);
    for (auto& t : th) t.join();
  }
  for (size_t i = 0; i < C; i++)
    if (bad[i]) {
      *err = 3;
      return nullptr;
    }
  d->d_l_u32.alloc(c, nl);
  d->d_m_u32.alloc(c, nm);
  d->d_l_fr.alloc(c, nl);
  d->d_m_fr.alloc(c, nm);
  LB_CUDA_CHECK(cudaMemcpyAsync(d->d_l_u32.p, l_host, nl * 4, cudaMemcpyHostToDevice, c->st));
  LB_CUDA_CHECK(cudaMemcpyAsync(d->d_m_u32.p, m_host, nm * 4, cudaMemcpyHostToDevice, c->st));
  launch_from_u32(d->d_l_u32.p, d->d_l_fr.p, nl, c->st);  // DensePolynomial::from_usize + merge
  launch_from_u32(d->d_m_u32.p, d->d_m_fr.p, nm, c->st);
  g_launches += 2;
  c->sync();
  return d.release();
}

// densified.rs:21-75 on an index matrix the caller already holds on the context's device (any of four integer types,
// element strides >= 0).  Ordered after the work queued on `producer`; returns once the extract has read the matrix
// and the range verdict is on the host (the sort and the field conversion stay queued).  Sharded: collective, every
// rank passes the same matrix on its own device, extracts its shard and checks every element itself.
Dense* densify_device(Ctx* c, const void* d_idx, int dtype, size_t n, size_t C, int64_t row_stride, int64_t col_stride,
                      size_t log_m, cudaStream_t producer, int* err) {
  SpanTimer sp(c, "Densify");
  std::unique_ptr<Dense> d = dense_header(c, n, C, log_m, err);
  if (!d) return nullptr;
  if (!densify_gpu_supported(d->s, log_m) || row_stride < 0 || col_stride < 0 || dtype < kDzU64 || dtype > kDzI32) {
    *err = 4;
    return nullptr;
  }
  cudaPointerAttributes pa;
  if (cudaPointerGetAttributes(&pa, d_idx) != cudaSuccess) {
    cudaGetLastError();  // an unknown pointer: clear the (non-sticky) error it left behind
    pa.type = cudaMemoryTypeUnregistered;
  }
  if (pa.type != cudaMemoryTypeDevice && pa.type != cudaMemoryTypeManaged)
    throw std::invalid_argument("densify_device: the indices are not device memory (host buffers go to lasso_densify)");
  if (pa.device != c->device)
    throw std::invalid_argument("densify_device: the indices are memory of device " + std::to_string(pa.device) +
                                ", the context is on device " + std::to_string(c->device));
  LB_CUDA_CHECK(cudaEventRecord(c->ev_input, producer));
  LB_CUDA_CHECK(cudaStreamWaitEvent(c->st, c->ev_input, 0));
  DBuf<uint32_t> bad(c, 1);
  LB_CUDA_CHECK(cudaMemsetAsync(bad.p, 0, 4, c->st));
  DzSource src;
  src.p = d_idx;
  src.type = dtype;
  src.row_stride = row_stride;
  src.col_stride = col_stride;
  src.bad = bad.p;
  src.bad_host = reinterpret_cast<uint32_t*>(c->h_pin);
  src.bad_ready = c->ev_aux;
  densify_on_device(c, d.get(), src, n);
  LB_CUDA_CHECK(cudaEventSynchronize(c->ev_aux));  // the extract is done: the caller's matrix is no longer read
  if (*src.bad_host) {
    *err = 3;
    return nullptr;  // d's arrays go back to the pool in stream order, behind the queued sort
  }
  return d.release();
}

// densified.rs:77-96 -> serialised SparsePolynomialCommitment (surge.rs:61-68)
std::vector<uint8_t> commit(Ctx* c, const Dense& d, const Gens& g) {
  SpanTimer sp(c, "DensifiedRepresentation.commit");
  if (g.nv_l != d.nv_l || g.nv_m != d.nv_m) throw std::runtime_error("generators were built for different (c, s, log_m)");
  unsigned bits = (unsigned)std::max(d.log_m, (size_t)(log2_exact_or_ceil(d.s) + 1));
  ByteWriter w;
  w.vec_pts(commit_u32(c, g, d.d_l_u32.p, d.nv_l, bits));
  w.vec_pts(commit_u32(c, g, d.d_m_u32.p, d.nv_m, bits));
  w.u64(d.s);
  w.u64(d.log_m);
  w.u64(d.m);
  return w.b;
}

// ---------------------------------------------------------------------------------------------- UniPoly
// unipoly.rs:30-54: coefficients of the polynomial through (0, e_0) .. (n-1, e_{n-1}).  The solution of the
// Vandermonde system is unique, so it is computed with a cached inverse matrix instead of eliminating
// per round.
static const std::vector<fr_t>& inv_vandermonde(size_t n) {
  static std::map<size_t, std::vector<fr_t>> cache;  // shared by every context of the process: guarded
  static std::mutex mu;
  std::lock_guard<std::mutex> lock(mu);  // (std::map never moves its nodes: the returned reference stays valid)
  auto it = cache.find(n);
  if (it != cache.end()) return it->second;
  std::vector<fr_t> a(n * 2 * n, fr_zero());  // [V | I], Gauss-Jordan
  for (size_t i = 0; i < n; i++) {
    fr_t x = fr_from_u64(i), p = fr_one();
    for (size_t j = 0; j < n; j++) {
      a[i * 2 * n + j] = p;
      p = fr_mul(p, x);
    }
    a[i * 2 * n + n + i] = fr_one();
  }
  for (size_t col = 0; col < n; col++) {
    size_t piv = col;
    while (fr_is_zero(a[piv * 2 * n + col])) piv++;
    if (piv != col)
      for (size_t k = 0; k < 2 * n; k++) std::swap(a[piv * 2 * n + k], a[col * 2 * n + k]);
    fr_t inv = fr_inv(a[col * 2 * n + col]);
    for (size_t k = 0; k < 2 * n; k++) a[col * 2 * n + k] = fr_mul(a[col * 2 * n + k], inv);
    for (size_t row = 0; row < n; row++) {
      if (row == col) continue;
      fr_t f = a[row * 2 * n + col];
      if (fr_is_zero(f)) continue;
      for (size_t k = 0; k < 2 * n; k++) a[row * 2 * n + k] = fr_sub(a[row * 2 * n + k], fr_mul(f, a[col * 2 * n + k]));
    }
  }
  std::vector<fr_t> inv(n * n);
  for (size_t i = 0; i < n; i++)
    for (size_t j = 0; j < n; j++) inv[i * n + j] = a[i * 2 * n + n + j];
  return cache[n] = inv;
}
static std::vector<fr_t> unipoly_from_evals(const std::vector<fr_t>& evals) {
  size_t n = evals.size();
  const std::vector<fr_t>& inv = inv_vandermonde(n);
  std::vector<fr_t> coeffs(n, fr_zero());
  for (size_t i = 0; i < n; i++)
    for (size_t j = 0; j < n; j++) coeffs[i] = fr_add(coeffs[i], fr_mul(inv[i * n + j], evals[j]));
  return coeffs;
}
static fr_t unipoly_evaluate(const std::vector<fr_t>& coeffs, const fr_t& r) {  // unipoly.rs:72-80
  fr_t eval = coeffs[0], power = r;
  for (size_t i = 1; i < coeffs.size(); i++) {
    eval = fr_add(eval, fr_mul(power, coeffs[i]));
    power = fr_mul(power, r);
  }
  return eval;
}
static void unipoly_append(const std::vector<fr_t>& coeffs, Transcript& t) {  // unipoly.rs:112-120
  t.append_message("poly", std::string("UniPoly_begin"));
  for (auto& cf : coeffs) t.append_scalar("coeff", cf);
  t.append_message("poly", std::string("UniPoly_end"));
}
typedef std::vector<std::vector<fr_t>> SumcheckProof;  // compressed polys: coeffs without the linear term
static std::vector<fr_t> unipoly_compress(const std::vector<fr_t>& coeffs) {  // unipoly.rs:82-88
  std::vector<fr_t> c;
  c.push_back(coeffs[0]);
  for (size_t i = 2; i < coeffs.size(); i++) c.push_back(coeffs[i]);
  return c;
}
static void ser_sumcheck(ByteWriter& w, const SumcheckProof& p) {
  w.u64(p.size());
  for (auto& c : p) w.vec_fr(c);
}

// ---------------------------------------------------------------------------------------------- sumcheck
// sumcheck.rs:149-260 over device polynomials W_k = base + k*stride (k <= alpha, the last is eq); `len_loc` is
// this rank's length.  Sharded rounds: local eval -> every rank's partial sums to every host (tagged publication
// into the shared host segments), added there; local bind.  When one element per rank is left the G-element
// remainders are all-gathered and the last log2(G) rounds run replicated.
static SumcheckProof prove_arbitrary(Ctx* c, const Strategy& S, fr_t* base, size_t stride, size_t len_loc,
                                     Transcript& transcript, std::vector<fr_t>& r) {
  SpanTimer sp(c, "Sumcheck.prove");
  SumcheckProof proof;
  r.clear();
  const int npts = S.sumcheck_poly_degree() + 1, npolys = S.num_memories() + 1;
  std::vector<fr_t> evals(npts);
  DBuf<fr_t> tail;
  bool sharded = c->world > 1;
  size_t len = len_loc;
  // The bind of a round is deferred into the next round's evaluation launch where the strategy has a fused kernel
  // (one pass over the polynomials per round instead of two); `pending` = the polynomials still have length 2*len
  const bool unfused = getenv("LASSO_B200_UNFUSED_PRIMARY") != nullptr;  // read per proof: A/B runs in one process
  bool pending = false;
  fr_t r_pending = fr_zero();
  auto flush_bind = [&]() {
    if (!pending) return;
    launch_bind_top(base, stride, npolys, len, r_pending, c->st);
    g_launches += 1;
    pending = false;
  };
  for (;;) {
    if (sharded && len == 1) {  // hand over to the replicated tail
      flush_bind();
      tail.alloc(c, (size_t)npolys * c->world);
      comm_gather_heads(c, nullptr, base, stride, npolys, nullptr, tail.p);
      base = tail.p;
      stride = (size_t)c->world;
      len = (size_t)c->world;
      sharded = false;
    }
    if (len <= 1) break;
    size_t half = len / 2;
    {  // sharded: every rank's partial sums go to every process, the hosts add them; else this process only
      Finalize f = c->fin_begin(sharded);
      if (pending && launch_sumcheck_bind_eval_arbitrary(S, base, stride, half, r_pending, f, 0, c->st)) {
        pending = false;
      } else {
        flush_bind();
        launch_sumcheck_eval_arbitrary(S, base, stride, half, f, c->st);
      }
      if (f.pub.ndst)
        c->fin_wait(f, evals.data(), npts);
      else
        c->d2h(evals.data(), c->d_small, (size_t)npts * sizeof(fr_t));
    }
    g_launches += 1;
    std::vector<fr_t> coeffs = unipoly_from_evals(evals);
    unipoly_append(coeffs, transcript);
    fr_t r_j = transcript.challenge_scalar("challenge_nextround");
    r.push_back(r_j);
    proof.push_back(unipoly_compress(coeffs));
    len = half;
    pending = true;
    r_pending = r_j;
    if (unfused) flush_bind();
  }
  flush_bind();
  return proof;
}

// ---------------------------------------------------------------------------------------------- grand products
// GrandProductCircuit (grand_product.rs:14-66): layer k is one contiguous array of N/2^k elements,
// left_vec[k] = first half, right_vec[k] = second half; layer k+1[i] = layer k[i] * layer k[i + N/2^(k+1)].
// Sharded: layers with N/2^k >= G are held as low-bit shards (local length N/(2^k G)); the layer of global
// length G is all-gathered and the few layers above it are kept replicated on every rank.
struct Circuit {
  DBuf<fr_t> tree;   // local shards: layer 0 at 0 (N/G elements), layer 1 after it, ...
  fr_t* rtree = nullptr;  // replicated top: layer k_rep (G elements), k_rep + 1, ... (2G slots in a shared allocation; G > 1)
  size_t N = 0, num_layers = 0;
  int G = 1;
  size_t k_rep = 0;  // first replicated layer: N >> k_rep == G
  bool layer_is_sharded(size_t k) const { return G == 1 || (N >> k) >= 2 * (size_t)G; }
  size_t layer_len_global(size_t k) const { return N >> k; }
  fr_t* layer_local(size_t k) const {  // valid for (N >> k) >= G
    size_t off = 0, len = N / G;
    for (size_t i = 0; i < k; i++) {
      off += len;
      len /= 2;
    }
    return tree.p + off;
  }
  fr_t* layer_rep(size_t k) const {  // valid for k >= k_rep (G > 1)
    size_t off = 0, len = (size_t)G;
    for (size_t i = k_rep; i < k; i++) {
      off += len;
      len /= 2;
    }
    return rtree + off;
  }
};
static void circuit_alloc(Ctx* c, Circuit& ci, size_t N, fr_t* rtree_slot) {
  ci.N = N;
  ci.G = c->world;
  ci.num_layers = log2_exact_or_ceil(N);
  ci.tree.alloc(c, 2 * (N / ci.G));
  if (ci.G > 1) {
    ci.k_rep = ci.num_layers - (size_t)c->lg_world;
    ci.rtree = rtree_slot;
  }
}
static void build_tree(Ctx* c, Circuit& ci) {  // grand_product.rs:38-58 (layer 0 already filled); single GPU, tree by tree
  for (size_t k = 0; k + 1 < ci.num_layers; k++) {
    launch_product_layer(ci.layer_local(k), ci.layer_local(k + 1), ci.layer_len_global(k + 1), c->st);
    g_launches += 1;
  }
}
// All product trees, size by size, layer by layer in batched launches (poly_kernels.cu).  groups[i] = trees of one
// (global) size sizes[i]; tops[i][2t], tops[i][2t+1] = the two elements of tree t's top layer (grand_product.rs:60-65
// `evaluate`).  Sharded: every rank builds the layers of its low-bit shard down to ONE element per tree (the layer
// of global length G), publishes it to every process, and each host computes the lg G layers above it — they are
// needed on the device too (the top layers of the grand-product argument run replicated): rtree_host mirrors the
// circuits' rtree slots and is uploaded by the caller.
static void build_trees(Ctx* c, std::vector<std::vector<Circuit*>>& groups, const std::vector<size_t>& sizes,
                        std::vector<std::vector<fr_t>>& tops, std::vector<fr_t>& rtree_host, const fr_t* rtree_base) {
  const int G = c->world;
  struct Pending {
    Finalize f;
    size_t grp, t0;
    int nt;
  };
  std::vector<Pending> pend;
  for (size_t gi = 0; gi < groups.size(); gi++) {
    tops[gi].assign(2 * groups[gi].size(), fr_zero());
    for (size_t t0 = 0; t0 < groups[gi].size(); t0 += 32) {
      const int nt = (int)std::min<size_t>(32, groups[gi].size() - t0);
      TreePtrs tp;
      for (int t = 0; t < nt; t++) tp.p[t] = groups[gi][t0 + t]->tree.p;
      if (pend.size() >= (size_t)kPubRegions) throw std::runtime_error("too many product-tree batches in flight");
      Finalize f = c->fin_begin(G > 1);
      launch_product_trees(tp, nt, sizes[gi] / (size_t)G, 0, G == 1 ? 2 : 1, f, c->st);
      g_launches += product_trees_launches(sizes[gi] / (size_t)G);
      pend.push_back({f, gi, t0, nt});
    }
  }
  for (auto& pd : pend) {
    fr_t* tp = tops[pd.grp].data() + 2 * pd.t0;
    if (G == 1) {
      c->fin_wait(pd.f, tp, 2 * pd.nt);
      continue;
    }
    std::vector<fr_t> rep((size_t)G * pd.nt);  // [rank][tree]: element `rank` of the layer of global length G
    for (int w = 0; w < G; w++) c->pub_wait_raw(pd.f.pub, w, pd.nt, (uint32_t*)(rep.data() + (size_t)w * pd.nt));
    for (int t = 0; t < pd.nt; t++) {
      Circuit& ci = *groups[pd.grp][pd.t0 + t];
      fr_t* h = rtree_host.data() + (ci.rtree - rtree_base);
      for (int w = 0; w < G; w++) h[w] = rep[(size_t)w * pd.nt + t];
      size_t off = 0, len = (size_t)G;
      while (len > 2) {  // layer k+1[i] = layer k[i] * layer k[i + len/2]
        for (size_t i = 0; i < len / 2; i++) h[off + len + i] = fr_mul(h[off + i], h[off + len / 2 + i]);
        off += len;
        len /= 2;
      }
      tp[2 * t] = h[off];
      tp[2 * t + 1] = h[off + 1];
    }
  }
}

struct LayerProof {
  SumcheckProof proof;
  std::vector<fr_t> claims_prod_left, claims_prod_right;
};
typedef std::vector<LayerProof> GPAProof;

// BatchedGrandProductArgument::prove (grand_product.rs:100-201) with prove_cubic_batched (sumcheck.rs:26-135)
static GPAProof prove_gpa(Ctx* c, std::vector<Circuit*>& circuits, std::vector<fr_t> claims_to_verify,
                          Transcript& transcript, std::vector<fr_t>& rand_out) {
  SpanTimer sp(c, "BatchedGrandProductArgument.prove");
  GPAProof out;
  const int ncirc = (int)circuits.size(), G = c->world;
  const size_t num_layers = circuits[0]->num_layers;
  // pointer tables: slot L (< num_layers) = the arrays of layer L, slot num_layers = the replicated tail arrays;
  // all of them are uploaded once, up front (no per-layer copy + sync)
  const size_t nslots = num_layers + 1;
  DBuf<fr_t*> d_ptrs(c, nslots * 4 * ncirc);
  const size_t eq_cap = std::max<size_t>(circuits[0]->N / 2 / G, (size_t)G);
  DBuf<fr_t> eqbuf(c, eq_cap), eqbuf2(c, std::max<size_t>(eq_cap / 2, 1));
  DBuf<fr_t> tail(c, (size_t)(2 * ncirc + 1) * G);  // replicated remainders of A_k, B_k, C (G elements each)
  std::vector<fr_t> rand;
  if (ncirc > 32) throw std::runtime_error("more than 32 circuits in one batched grand product");
  std::vector<fr_t> ev(3), fin((size_t)2 * ncirc);
  // per slot: [A_0..A_{n-1} | B_0..B_{n-1} | A_0,B_0,A_1,B_1,...]
  std::vector<fr_t*> table(nslots * 4 * ncirc);
  auto slot_A = [&](size_t slot) { return d_ptrs.p + slot * 4 * ncirc; };
  auto slot_B = [&](size_t slot) { return d_ptrs.p + slot * 4 * ncirc + ncirc; };
  auto slot_AB = [&](size_t slot) { return d_ptrs.p + slot * 4 * ncirc + 2 * ncirc; };
  auto layer_cur = [&](size_t layer_id, bool& replicated_layer) {
    const size_t len_g = circuits[0]->layer_len_global(layer_id);
    replicated_layer = G > 1 && !circuits[0]->layer_is_sharded(layer_id);
    return replicated_layer ? len_g / 2 : len_g / 2 / (size_t)G;  // |A| = |B| = |C| on this rank
  };
  for (size_t slot = 0; slot < nslots; slot++) {
    for (int k = 0; k < ncirc; k++) {
      fr_t *pa, *pb;
      if (slot == num_layers) {
        pa = tail.p + (size_t)(2 * k) * G;
        pb = tail.p + (size_t)(2 * k + 1) * G;
      } else {
        bool rep;
        size_t cur0 = layer_cur(slot, rep);
        pa = rep ? circuits[k]->layer_rep(slot) : circuits[k]->layer_local(slot);
        pb = pa + cur0;
      }
      table[slot * 4 * ncirc + k] = pa;
      table[slot * 4 * ncirc + ncirc + k] = pb;
      table[slot * 4 * ncirc + 2 * ncirc + 2 * k] = pa;
      table[slot * 4 * ncirc + 2 * ncirc + 2 * k + 1] = pb;
    }
  }
  LB_CUDA_CHECK(cudaMemcpyAsync(d_ptrs.p, table.data(), table.size() * sizeof(fr_t*), cudaMemcpyHostToDevice, c->st));
  c->sync();
  for (size_t layer_id = num_layers; layer_id-- > 0;) {
    bool replicated_layer;
    size_t cur = layer_cur(layer_id, replicated_layer);
    bool sharded = G > 1 && !replicated_layer;
    fr_t* const* dA = slot_A(layer_id);
    fr_t* const* dB = slot_B(layer_id);
    fr_t* const* dAB = slot_AB(layer_id);
    // poly_C = eq(rand), grand_product.rs:122
    if (sharded)
      eq_evals_shard(c, rand, 0, rand.size(), eqbuf.p);
    else
      eq_evals_dev(c, rand, 0, rand.size(), eqbuf.p);
    std::vector<fr_t> coeff_vec = transcript.challenge_vector("rand_coeffs_next_layer", ncirc);
    fr_t e = fr_zero();
    for (int k = 0; k < ncirc; k++) e = fr_add(e, fr_mul(claims_to_verify[k], coeff_vec[k]));
    // The kernels fold the batching coefficients in (poly_kernels.cu): the first bind of the layer stores
    // coeff_k * A_k, a round message is the 3 combined values of sumcheck.rs:95-97.
    CubicCoeffs cf;
    for (int k = 0; k < ncirc; k++) cf.v[k] = coeff_vec[k];
    bool stored_scaled = false;
    std::vector<fr_t> inv_coeff;  // computed while the first kernel of the layer runs
    LayerProof lp;
    std::vector<fr_t> rand_prod;
    fr_t* Ccur = eqbuf.p;
    fr_t* Cnext = eqbuf2.p;
    bool have_evals = false, heads_published = false;
    Finalize fz = c->fin_begin();
    for (;;) {
      if (sharded && cur == 1) {  // all-gather the G-element remainders; the tail rounds run replicated
        comm_gather_heads(c, dAB, nullptr, 0, 2 * ncirc, Ccur, tail.p);  // A_k, B_k and eq in one exchange
        dA = slot_A(num_layers);
        dB = slot_B(num_layers);
        dAB = slot_AB(num_layers);
        Ccur = tail.p + (size_t)2 * ncirc * G;
        Cnext = eqbuf2.p;
        cur = (size_t)G;
        sharded = false;
        have_evals = false;
      }
      if (cur <= 1) break;
      if (!have_evals) {  // first round of a phase; later rounds come out of the fused bind+eval kernel
        fz = c->fin_begin(sharded);
        launch_sumcheck_eval_cubic_comb(dA, dB, Ccur, ncirc, cur / 2, cf, stored_scaled ? 0 : 1, fz, c->st);
        g_launches += 1;
      }
      if (inv_coeff.empty()) {  // 1 / coeff_k by Montgomery's trick, overlapping the kernel just launched
        inv_coeff.resize(ncirc);
        std::vector<fr_t> pre(ncirc);
        fr_t acc = fr_one();
        for (int k = 0; k < ncirc; k++) {
          pre[k] = acc;
          acc = fr_mul(acc, coeff_vec[k]);
        }
        if (fr_eq(acc, fr_zero())) throw std::runtime_error("zero batching coefficient");
        fr_t ainv = fr_inv(acc);
        for (int k = ncirc; k-- > 0;) {
          inv_coeff[k] = fr_mul(ainv, pre[k]);
          ainv = fr_mul(ainv, coeff_vec[k]);
        }
      }
      size_t half = cur / 2;
      auto tp0 = std::chrono::steady_clock::now();
      if (fz.pub.ndst)  // sharded: the three sums of every rank, added here
        c->fin_wait(fz, ev.data(), 3);
      else
        c->d2h(ev.data(), c->d_small, ev.size() * sizeof(fr_t));
      auto tp1 = std::chrono::steady_clock::now();
      const fr_t c0 = ev[0], c2 = ev[1], c3 = ev[2];  // already combined over the circuits (sumcheck.rs:95-97)
      std::vector<fr_t> evals = {c0, fr_sub(e, c0), c2, c3};  // eval(1) = e - eval(0), sumcheck.rs:99-104
      std::vector<fr_t> coeffs = unipoly_from_evals(evals);
      unipoly_append(coeffs, transcript);
      fr_t r_j = transcript.challenge_scalar("challenge_nextround");
      rand_prod.push_back(r_j);
      auto tp2 = std::chrono::steady_clock::now();
      if (half > 1) {
        // bind with r_j and evaluate the next round in one pass (sumcheck.rs:116-120 + 63-89)
        fz = c->fin_begin(sharded);
        launch_sumcheck_bind_eval_cubic_comb(dA, dB, Ccur, Cnext, ncirc, half, r_j, cf, stored_scaled ? 0 : 1, fz, c->st);
        stored_scaled = true;
        g_launches += 1;
        std::swap(Ccur, Cnext);
        have_evals = true;
      } else if (!sharded && fz.pub.ndst) {
        // last round: bind the 2*ncirc heads and publish them (the layer's claims); eq is not needed any more
        fz = c->fin_begin();
        launch_bind_heads(dAB, 2 * ncirc, r_j, fz, c->st);
        g_launches += 1;
        have_evals = false;
        heads_published = true;
      } else {
        launch_bind_top_ptrs(dAB, 2 * ncirc, half, r_j, c->st);
        launch_bind_top(Ccur, 0, 1, half, r_j, c->st);
        g_launches += 2;
        have_evals = false;
      }
      auto tp3 = std::chrono::steady_clock::now();
      if (c->span_sync) {  // where a grand-product round goes: waiting for the device, host glue, launch call
        c->spans["GPA.round wait"] += std::chrono::duration<double, std::milli>(tp1 - tp0).count();
        c->spans["GPA.round host"] += std::chrono::duration<double, std::milli>(tp2 - tp1).count();
        c->spans["GPA.round launch"] += std::chrono::duration<double, std::milli>(tp3 - tp2).count();
      }
      e = unipoly_evaluate(coeffs, r_j);
      lp.proof.push_back(unipoly_compress(coeffs));
      cur = half;
    }
    // claims_prod = (A_k[0], B_k[0]): published by the last round's kernel, or packed on the device + one transfer
    if (heads_published) {
      c->fin_wait(fz, fin.data(), 2 * ncirc);
    } else {
      pack_heads(c, dAB, nullptr, 0, 2 * ncirc, c->d_small + 1024);
      c->d2h(fin.data(), c->d_small + 1024, fin.size() * sizeof(fr_t));
    }
    for (int k = 0; k < ncirc; k++) {  // the left arrays carry coeff_k once a bind has stored them
      lp.claims_prod_left.push_back(stored_scaled ? fr_mul(fin[2 * k], inv_coeff[k]) : fin[2 * k]);
      lp.claims_prod_right.push_back(fin[2 * k + 1]);
    }
    for (int k = 0; k < ncirc; k++) {
      transcript.append_scalar("claim_prod_left", lp.claims_prod_left[k]);
      transcript.append_scalar("claim_prod_right", lp.claims_prod_right[k]);
    }
    fr_t r_layer = transcript.challenge_scalar("challenge_r_layer");
    for (int k = 0; k < ncirc; k++)
      claims_to_verify[k] = fr_add(lp.claims_prod_left[k],
                                   fr_mul(r_layer, fr_sub(lp.claims_prod_right[k], lp.claims_prod_left[k])));
    std::vector<fr_t> ext = {r_layer};
    ext.insert(ext.end(), rand_prod.begin(), rand_prod.end());
    rand = ext;
    out.push_back(std::move(lp));
  }
  rand_out = rand;
  return out;
}
static void ser_gpa(ByteWriter& w, const GPAProof& p) {
  w.u64(p.size());
  for (auto& l : p) {
    ser_sumcheck(w, l.proof);
    w.vec_fr(l.claims_prod_left);
    w.vec_fr(l.claims_prod_right);
  }
}

// ---------------------------------------------------------------------------------------------- openings
struct DotProductProofLogBytes {  // dot_product.rs:152-159 field order
  std::vector<uint8_t> L_vec, R_vec;  // 32 B per point
  uint8_t delta[32], beta[32];
  fr_t z1, z2;
};
static void ser_dpl(ByteWriter& w, const DotProductProofLogBytes& p) {
  w.vec_pts(p.L_vec);
  w.vec_pts(p.R_vec);
  w.raw(p.delta, 32);
  w.raw(p.beta, 32);
  w.fr(p.z1);
  w.fr(p.z2);
}

// dst (nrows x 2, row-major) <- [ip[0], blind_L ; ip[1], blind_R]
__global__ void set_tail_kernel(fr_t* dst0, fr_t* dst1, const fr_t* ip, fr_t blind_L, fr_t blind_R) {
  if (threadIdx.x || blockIdx.x) return;
  dst0[0] = ip[0];  // c_L on Q
  dst0[1] = blind_L;  // on H
  dst1[0] = ip[1];
  dst1[1] = blind_R;
}
__global__ void set_elems_kernel(fr_t* dst, fr_t a, fr_t b) {
  if (threadIdx.x || blockIdx.x) return;
  dst[0] = a;
  dst[1] = b;
}

// PolyEvalProof::prove (dense_mlpoly.rs:301-359) -> DotProductProofLog::prove (dot_product.rs:166-249)
// -> BulletReductionProof::prove (bullet.rs:40-154).  Z: this rank's shard of a polynomial of 2^nv elements,
// i.e. for every one of the L rows the R/G columns congruent to the rank.
// One proof sharded over G GPUs: LZ = L . Z is computed on the column shards and all-gathered (R elements); from
// there on the opening runs REPLICATED on every rank — its vectors are only R = 2^(nv - nv/2) long and every round
// is latency-bound, so splitting its two-row MSMs would add an exchange per round and save nothing.  Every rank
// computes the same points and the same transcript.
static DotProductProofLogBytes prove_poly_eval(Ctx* c, const Gens& g, const fr_t* Z, const uint32_t* Z_u32, size_t nv,
                                               const std::vector<fr_t>& r, const fr_t& Zr, Transcript& transcript,
                                               RandomTape& tape) {
  SpanTimer sp(c, "DensePolyEval.prove");
  transcript.append_protocol_name("polynomial evaluation proof");
  if (r.size() != nv) throw std::runtime_error("PolyEvalProof: r.len() != num_vars");
  const int G = c->world;
  const size_t lv = nv / 2, rv = nv - nv / 2, L_size = (size_t)1 << lv, n = (size_t)1 << rv;  // n = R_size
  if (n + 2 > g.n_points) throw std::runtime_error("generator stream too short");
  if (n < (size_t)G) throw std::runtime_error("opening narrower than the number of GPUs");
  const size_t lg_n = rv, n_loc = n / G;
  // L, R = factored eq evals (eq_poly.rs:44-52); LZ = L . Z (dense_mlpoly.rs:183-207)
  std::unique_ptr<SpanTimer> sp1(new SpanTimer(c, "PE.1 eq+bound"));
  DBuf<fr_t> Lvec(c, L_size), a(c, n), b(c, n), a_loc(c, G > 1 ? n_loc : 0), a_gath(c, G > 1 ? n : 0);
  eq_evals_dev(c, r, 0, lv, Lvec.p);  // rows are not sharded: L is replicated
  eq_evals_dev(c, r, lv, rv, b.p);    // a_vec of the dot product proof = R
  if ((size_t)bound_max_chunks() * n_loc > c->partial_elems) throw std::runtime_error("bound scratch too small");
  // x_vec = LZ (this rank's columns); the opened polynomials are integer-valued: over their u32 mirror when there is one
  if (Z_u32)
    launch_bound_u32(Z_u32, Lvec.p, L_size, n_loc, c->d_partial, G > 1 ? a_loc.p : a.p, c->st);
  else
    launch_bound(Z, Lvec.p, L_size, n_loc, c->d_partial, G > 1 ? a_loc.p : a.p, c->st);
  g_launches += 2;
  if (G > 1) comm_gather_vector(c, a_loc.p, n_loc, a_gath.p, a.p);

  // ---- DotProductProofLog::prove
  sp1.reset(new SpanTimer(c, "PE.2 Cx,Cy,append a"));
  transcript.append_protocol_name("dot product proof (log)");
  fr_t d = tape.random_scalar("d");
  fr_t r_delta = tape.random_scalar("r_delta");
  fr_t r_beta = tape.random_scalar("r_delta");  // sic (dot_product.rs:189)
  std::vector<fr_t> v1 = tape.random_vector("blinds_vec_1", 2 * lg_n);
  std::vector<fr_t> v2 = tape.random_vector("blinds_vec_2", 2 * lg_n);
  DotProductProofLogBytes out;
  // table pipeline below: needs the multiples table of the generators 0 .. n+1
  const bool fast = c->h_pub != nullptr && n * 32 <= c->h_pin_bytes && g.d_multiples.p && n + 2 <= g.n_direct;
  // ---- BulletReductionProof::prove with unfolded generators (see file header)
  fr_t blind_fin = fr_zero();  // blind_Gamma = blind_x + blind_y = 0
  DBuf<fr_t> W0(c, n), W1(c, n), sLR(c, 2 * (n + 2));
  fr_t* W = W0.p;   // weights of the unfolded generators (indexed by the HIGH column bits)
  fr_t* Wn = W1.p;
  set_elems_kernel<<<1, 32, 0, c->st>>>(W, fr_one(), fr_zero());
  LB_LAUNCH_CHECK();
  g_launches += 1;
  fr_t* sL = sLR.p;
  fr_t* sR = sLR.p + (n + 2);
  fr_t* av = a.p;  // current a / b vectors
  fr_t* bv = b.p;
  DBuf<fr_t> a_alt, b_alt;
  if (fast) {
    // Per message ONE scalar kernel + the two MSM kernels, the finish kernel publishing straight to mapped host
    // memory; the host part of a message (compression, Fiat-Shamir) overlaps the device work of the next one
    // wherever the transcript allows it.
    //   (Cx, Cy): rows (x_vec, 0, 0) and (0.., y, 0) of one two-row MSM        (dot_product.rs:192-197)
    //   round k : fold with u_{k-1}, weights, L/R scalars, c_L, c_R -> two-row MSM   (bullet.rs:73-134)
    auto read_two_points = [&](const PubDst& pd, uint8_t* comp64) {
      uint32_t xyz[48];
      c->wait_points(pd, 2, xyz);
      h64::compress_xyz_pair(xyz, xyz + 24, comp64, comp64 + 32);  // one Fq inversion for both points
    };
    a_alt.alloc(c, n);
    b_alt.alloc(c, n);
    fr_t *an = a_alt.p, *bn = b_alt.p;
    DBuf<pt_ext> part(c, 2 * (size_t)msm_direct_chunks((int)(n + 2), 1));
    DBuf<fr_t> canon(c, n);
    DBuf<uint32_t> cols(c, 2 * (n / 2 + 2));
    // two short rows over the multiples table; len terms per row, generator index per term in cols (or identity)
    // heavy = rows that carry the terms: both in a round (L, R), one for (Cx, Cy) — Cy is a single term
    auto two_row_msm = [&](const uint32_t* d_cols, size_t len, int heavy) {
      const PubDst pd = c->pub_begin(false);
      launch_msm_direct(g.d_multiples.p, g.n_direct, (const uint32_t*)sLR.p, d_cols, 2, (int)len, heavy, part.p, nullptr, pd,
                        c->st);
      g_launches += 2;
      return pd;
    };
    launch_two_row_scalars(av, 0, fr_one(), fr_zero(), fr_zero(), Zr, fr_zero(), n, sLR.p, c->st);
    const PubDst pd_c = two_row_msm(nullptr, n + 2, 1);
    // a_vec of the transcript = canonical bytes of b; the copy is waited for only when it is appended
    launch_canonicalize(bv, canon.p, n, c->d_flag, c->st);
    LB_CUDA_CHECK(cudaMemcpyAsync(c->h_pin, canon.p, n * 32, cudaMemcpyDeviceToHost, c->st));
    LB_CUDA_CHECK(cudaEventRecord(c->ev_aux, c->st));
    g_launches += 2;
    fr_t u = fr_one(), u_inv = fr_one();
    int fold = 0;
    size_t m = n;  // vector length entering the round (after the fold with the previous challenge)
    PubDst pd_round;
    static const bool unfused = [] {
      const char* e = getenv("LASSO_B200_UNFUSED_ROUNDS");
      return e && e[0] == '1';
    }();
    DBuf<pt_ext> part_f(c, 2 * (size_t)bullet_fused_chunks((int)n));
    auto launch_round = [&](size_t round) {
      if (!unfused) {
        // the whole round in ONE launch: scalars, both rows over the multiples table, tail terms, publication
        pd_round = c->pub_begin(false);
        launch_bullet_fused(g.d_multiples.p, g.n_direct, av, bv, W, an, bn, Wn, n, m, fold, u, u_inv, v1[round], v2[round],
                            part_f.p, c->d_partial, c->d_flag + 4, pd_round, c->st);
        g_launches += 1;
      } else {
        launch_bullet_round(av, bv, W, an, bn, Wn, n, m, fold, u, u_inv, v1[round], v2[round], sLR.p, cols.p, c->d_partial,
                            c->d_flag + 4, c->st);
        g_launches += 1;
      }
      if (fold) {
        std::swap(av, an);
        std::swap(bv, bn);
        std::swap(W, Wn);
      }
      if (unfused) pd_round = two_row_msm(cols.p, n / 2 + 2, 2);
    };
    // NB: the (Cx, Cy) MSM reads sLR before round 0 overwrites it: same stream, so ordered
    uint8_t CxCy[64];
    read_two_points(pd_c, CxCy);
    if (m != 1) launch_round(0);  // round 0 needs no challenge: it runs while the host absorbs Cx, Cy, a
    transcript.append_point_compressed("Cx", CxCy);
    transcript.append_point_compressed("Cy", CxCy + 32);
    LB_CUDA_CHECK(cudaEventSynchronize(c->ev_aux));
    transcript.append_scalars_bytes("a", c->h_pin, n);
    sp1.reset(new SpanTimer(c, "PE.3 bullet rounds"));
    for (size_t round = 0; m != 1; round++) {
      uint8_t LR[64];
      read_two_points(pd_round, LR);
      transcript.append_point_compressed("L", LR);
      transcript.append_point_compressed("R", LR + 32);
      u = transcript.challenge_scalar("u");
      u_inv = fr_inv(u);
      fold = 1;
      m /= 2;
      if (m != 1) launch_round(round + 1);
      blind_fin = fr_add(blind_fin, fr_add(fr_mul(fr_mul(v1[round], u), u), fr_mul(fr_mul(v2[round], u_inv), u_inv)));
      out.L_vec.insert(out.L_vec.end(), LR, LR + 32);
      out.R_vec.insert(out.R_vec.end(), LR + 32, LR + 64);
    }
    if (fold) {  // the last challenge: a, b -> one element each, weights -> n (bullet.rs:127-134)
      launch_fold_ab(av, bv, 1, u, u_inv, c->st);
      launch_expand_weights(W, Wn, n / 2, u, u_inv, c->st);
      g_launches += 2;
      std::swap(W, Wn);
    }
  } else {
    // no multiples table (LASSO_B200_NO_MULTIPLES=1 / not enough memory) or no mapped buffers: bucket MSMs over
    // the window table, one kernel per step
    DBuf<fr_t> two(c, 4);
    {
      // Cx = batch_commit(x_vec, blind_x = 0) ; Cy = y*Q + 0*h
      std::vector<uint8_t> Cx = msm_rows_fr(c, g, a.p, 1, (int)n);
      transcript.append_point_compressed("Cx", Cx.data());
      // (0 .. 0, y, 0) on (G_0 .. G_{n-1}, Q, h)
      launch_fill_zero(sL, n, c->st);
      set_elems_kernel<<<1, 32, 0, c->st>>>(sL + n, Zr, fr_zero());
      LB_LAUNCH_CHECK();
      g_launches += 1;
      std::vector<uint8_t> Cy = msm_rows_fr(c, g, sL, 1, (int)(n + 2));
      transcript.append_point_compressed("Cy", Cy.data());
      // append_scalars(b"a", a_vec): canonical bytes straight from the device
      DBuf<fr_t> canon(c, n);
      launch_canonicalize(b.p, canon.p, n, c->d_flag, c->st);
      g_launches += 1;
      std::vector<uint8_t> bytes(n * 32);
      c->d2h(bytes.data(), canon.p, bytes.size());
      transcript.append_scalars_bytes("a", bytes.data(), n);
    }
    sp1.reset(new SpanTimer(c, "PE.3 bullet rounds"));
    size_t m = n, nw_count = 1;  // current vector length, number of weights
    for (size_t round = 0; m != 1; round++) {
      const size_t h = m / 2;
      launch_cross_inner_products(av, bv, h, c->d_partial, c->d_small, c->st);  // c_L, c_R (bullet.rs:78-79)
      g_launches += 2;
      launch_bullet_scalars(av, W, n, m, 1, 0, 0, sL, sR, c->st);
      set_tail_kernel<<<1, 32, 0, c->st>>>(sL + n, sR + n, c->d_small, v1[round], v2[round]);
      LB_LAUNCH_CHECK();
      g_launches += 2;
      std::vector<uint8_t> LR = msm_rows_fr(c, g, sLR.p, 2, (int)(n + 2));
      transcript.append_point_compressed("L", LR.data());
      transcript.append_point_compressed("R", LR.data() + 32);
      fr_t u = transcript.challenge_scalar("u");
      fr_t u_inv = fr_inv(u);
      launch_fold_ab(av, bv, h, u, u_inv, c->st);  // bullet.rs:127-130 (scalars only; G stays unfolded)
      launch_expand_weights(W, Wn, nw_count, u, u_inv, c->st);
      g_launches += 2;
      std::swap(W, Wn);
      nw_count *= 2;
      blind_fin = fr_add(blind_fin, fr_add(fr_mul(fr_mul(v1[round], u), u), fr_mul(fr_mul(v2[round], u_inv), u_inv)));
      out.L_vec.insert(out.L_vec.end(), LR.begin(), LR.begin() + 32);
      out.R_vec.insert(out.R_vec.end(), LR.begin() + 32, LR.begin() + 64);
      m = h;
    }
  }
  sp1.reset(new SpanTimer(c, "PE.4 delta,beta"));
  fr_t ab[2];
  if (fast) {
    // delta = d * g_hat + r_delta * h with g_hat = sum_j W[j] G_j (dot_product.rs:219-227) and
    // beta = d * Q + r_beta * h (dot_product.rs:229-230) as the two rows of one MSM
    launch_two_row_scalars(W, 1, d, fr_zero(), r_delta, d, r_beta, n, sLR.p, c->st);
    DBuf<pt_ext> part(c, 2 * (size_t)msm_direct_chunks((int)(n + 2), 1));
    const PubDst pd = c->pub_begin(false);
    launch_msm_direct(g.d_multiples.p, g.n_direct, (const uint32_t*)sLR.p, nullptr, 2, (int)(n + 2), 1, part.p, nullptr, pd,
                      c->st);
    LB_CUDA_CHECK(cudaMemcpyAsync(c->h_pin, av, 32, cudaMemcpyDeviceToHost, c->st));
    LB_CUDA_CHECK(cudaMemcpyAsync(c->h_pin + 32, bv, 32, cudaMemcpyDeviceToHost, c->st));
    g_launches += 3;
    uint32_t xyz[48];
    c->wait_points(pd, 2, xyz);
    h64::compress_xyz_pair(xyz, xyz + 24, out.delta, out.beta);
    c->sync();
    memcpy(ab, c->h_pin, 64);
    transcript.append_point_compressed("delta", out.delta);
    transcript.append_point_compressed("beta", out.beta);
  } else {
    LB_CUDA_CHECK(cudaMemcpyAsync(c->h_pin, av, 32, cudaMemcpyDeviceToHost, c->st));
    LB_CUDA_CHECK(cudaMemcpyAsync(c->h_pin + 32, bv, 32, cudaMemcpyDeviceToHost, c->st));
    c->sync();
    memcpy(ab, c->h_pin, 64);
    // delta = d * g_hat + r_delta * h with g_hat = sum_j W[j] G_j  (dot_product.rs:219-227)
    launch_scale(W, sL, n, d, c->st);
    set_elems_kernel<<<1, 32, 0, c->st>>>(sL + n, fr_zero(), r_delta);
    LB_LAUNCH_CHECK();
    g_launches += 2;
    std::vector<uint8_t> delta = msm_rows_fr(c, g, sL, 1, (int)(n + 2));
    memcpy(out.delta, delta.data(), 32);
    transcript.append_point_compressed("delta", out.delta);
    // beta = d * Q + r_beta * h  (dot_product.rs:229-230)
    launch_fill_zero(sL, n, c->st);
    set_elems_kernel<<<1, 32, 0, c->st>>>(sL + n, d, r_beta);
    LB_LAUNCH_CHECK();
    g_launches += 1;
    std::vector<uint8_t> beta = msm_rows_fr(c, g, sL, 1, (int)(n + 2));
    memcpy(out.beta, beta.data(), 32);
    transcript.append_point_compressed("beta", out.beta);
  }
  fr_t x_hat = ab[0], a_hat = ab[1], rhat_Gamma = blind_fin;
  fr_t y_hat = fr_mul(x_hat, a_hat);
  fr_t cc = transcript.challenge_scalar("c");
  out.z1 = fr_add(d, fr_mul(cc, y_hat));
  out.z2 = fr_add(fr_mul(a_hat, fr_add(fr_mul(cc, rhat_Gamma), r_beta)), r_delta);
  return out;
}

// CombinedTableEvalProof::prove (subtables/mod.rs:284-313 + prove_single 230-281) and the two analogous
// n-to-1 reductions of HashLayerProof::prove: fold `evals` with bound_poly_var_bot in reverse challenge order.
static DotProductProofLogBytes prove_joint(Ctx* c, const Gens& g, const fr_t* Z, const uint32_t* Z_u32, size_t nv, std::vector<fr_t> evals,
                                           bool pad_before_append, const char* evals_label, const char* chal_label,
                                           const char* joint_label, const std::vector<fr_t>& r,
                                           Transcript& transcript, RandomTape& tape) {
  std::vector<fr_t> padded = evals;
  padded.resize(next_pow2(padded.size()), fr_zero());
  if (pad_before_append) evals = padded;
  transcript.append_scalars(evals_label, evals.data(), evals.size());
  std::vector<fr_t> challenges = transcript.challenge_vector(chal_label, log2_exact_or_ceil(evals.size()));
  std::vector<fr_t> pe = padded;
  for (size_t i = challenges.size(); i-- > 0;) {  // bound_poly_var_bot (dense_mlpoly.rs:218-225), tiny: host
    size_t half = pe.size() / 2;
    for (size_t k = 0; k < half; k++)
      pe[k] = fr_add(pe[2 * k], fr_mul(challenges[i], fr_sub(pe[2 * k + 1], pe[2 * k])));
    pe.resize(half);
  }
  fr_t joint = pe[0];
  std::vector<fr_t> r_joint = challenges;
  r_joint.insert(r_joint.end(), r.begin(), r.end());
  transcript.append_scalar(joint_label, joint);
  return prove_poly_eval(c, g, Z, Z_u32, nv, r_joint, joint, transcript, tape);
}

// ---------------------------------------------------------------------------------------------- prove
std::vector<uint8_t> prove(Ctx* c, const Strategy& S, Dense& dense, const std::vector<fr_t>& r, const Gens& g,
                           const std::string& transcript_label, const std::string& tape_label, const fr_t& tape_seed,
                           std::vector<fr_t>* challenges) {
  SpanTimer sp_all(c, "SparsePoly.prove");
  Transcript transcript(transcript_label);
  transcript.trace = challenges;
  RandomTape tape(tape_label, tape_seed);
  const int G = c->world, gr = c->rank;
  const size_t s = dense.s, C = dense.C, M = dense.m, alpha = (size_t)S.num_memories();
  const size_t s_loc = dense.s_loc, M_loc = dense.m_loc;
  const size_t log_s = log2_exact_or_ceil(s);
  if ((size_t)S.C != C || (size_t)S.log_m != dense.log_m) throw std::runtime_error("strategy does not match the densified representation");
  if (g.nv_d != log2_exact_or_ceil(next_pow2(alpha * s)) || g.nv_l != dense.nv_l || g.nv_m != dense.nv_m)
    throw std::runtime_error("generators were built for different (c, s, num_memories, log_m)");
  transcript.append_protocol_name("Lasso SparsePolynomialEvaluationProof");

  // ---- Subtables::new (subtables/mod.rs:116-129): materialise (replicated, 2-6 MiB), gather, merge
  const size_t nv_d = g.nv_d, nd_loc = ((size_t)1 << nv_d) / G;
  const int nsub = S.num_subtables();
  DBuf<fr_t> tables_fr(c, (size_t)nsub * M);
  DBuf<uint32_t> tables_u32(c, (size_t)nsub * M);
  DBuf<fr_t> E(c, nd_loc);          // combined_poly = E_0 | .. | E_{alpha-1} | 0-pad (this rank's shard)
  DBuf<uint32_t> E_u32(c, nd_loc);  // same values as integers for the small-scalar commit
  {
    SpanTimer sp(c, "Subtables.new");
    launch_materialize_subtables(S, tables_fr.p, tables_u32.p, c->st);
    launch_gather_lookup_polys(S, tables_fr.p, tables_u32.p, dense.nz(), s_loc, E.p, s_loc, E_u32.p, c->st);
    g_launches += 2;
    if (nd_loc > alpha * s_loc) {
      launch_fill_zero(E.p + alpha * s_loc, nd_loc - alpha * s_loc, c->st);
      LB_CUDA_CHECK(cudaMemsetAsync(E_u32.p + alpha * s_loc, 0, (nd_loc - alpha * s_loc) * 4, c->st));
    }
  }
  ByteWriter w;
  std::vector<uint8_t> comm_E;
  // ---- comm_derefs (surge.rs:136-140, subtables/mod.rs:177-184, 382-393)
  {
    SpanTimer sp(c, "Subtables.commit");
    unsigned tbits = S.kind == STRAT_LT ? 1 : (S.kind == STRAT_RANGE ? (unsigned)S.log_m : (unsigned)(S.log_m / 2));
    comm_E = commit_u32(c, g, E_u32.p, nv_d, tbits);
    w.vec_pts(comm_E);
  }
  auto absorb_comm_E = [&]() {  // ~700 Keccak permutations (2^11 points): done while the device prepares the sumcheck
    transcript.append_message("subtable_evals_commitment", std::string("begin_subtable_evals_commitment"));
    transcript.append_message("comm_poly_row_col_ops_val", std::string("poly_commitment_begin"));
    for (size_t i = 0; i < comm_E.size() / 32; i++)
      transcript.append_point_compressed("poly_commitment_share", comm_E.data() + 32 * i);
    transcript.append_message("comm_poly_row_col_ops_val", std::string("poly_commitment_end"));
    transcript.append_message("subtable_evals_commitment", std::string("end_subtable_evals_commitment"));
  };
  // ---- primary sumcheck (surge.rs:142-172)
  std::vector<fr_t> r_z;
  {
    DBuf<fr_t> Wk(c, (alpha + 1) * s_loc);  // clones of E_i + eq(r): the sumcheck binds them in place
    LB_CUDA_CHECK(cudaMemcpyAsync(Wk.p, E.p, alpha * s_loc * sizeof(fr_t), cudaMemcpyDeviceToDevice, c->st));
    eq_evals_shard(c, r, 0, log_s, Wk.p + alpha * s_loc);
    launch_sumcheck_claim(S, Wk.p, s_loc, s_loc, c->d_partial, c->d_small, c->st);  // subtables/mod.rs:186-216
    g_launches += 2;
    fr_t claimed_eval;
    const Finalize fclaim = reduce_to_host_begin(c, c->d_small, 1);
    absorb_comm_E();  // transcript order unchanged: the commitment, then the claim
    reduce_to_host_end(c, fclaim, c->d_small, 1, &claimed_eval);
    transcript.append_scalar("claim_eval_scalar_product", claimed_eval);
    SumcheckProof primary = prove_arbitrary(c, S, Wk.p, s_loc, s_loc, transcript, r_z);
    ser_sumcheck(w, primary);
    w.fr(claimed_eval);
  }
  // ---- eval_derefs = E_i(r_z) (surge.rs:175-176) and the combined opening (177-184)
  DBuf<fr_t> eqtab(c, std::max(s_loc, M_loc));
  std::vector<fr_t> eval_derefs(alpha);
  {
    SpanTimer sp(c, "CombinedEval.prove");
    eq_evals_shard(c, r_z, 0, log_s, eqtab.p);
    launch_multi_dot_u32(E_u32.p, s_loc, (int)alpha, eqtab.p, s_loc, c->d_partial, c->d_small, c->st);
    g_launches += 2;
    reduce_to_host(c, c->d_small, (int)alpha, eval_derefs.data());
    w.arr_fr(eval_derefs);
    transcript.append_protocol_name("Lasso CombinedTableEvalProof");
    ser_dpl(w, prove_joint(c, g, E.p, E_u32.p, nv_d, eval_derefs, true, "evals_ops_val", "challenge_combine_n_to_one",
                           "joint_claim_eval", r_z, transcript, tape));
  }
  // ---- memory checking (surge.rs:186-198)
  std::vector<fr_t> r_hash = transcript.challenge_vector("challenge_r_hash", 2);
  const fr_t gamma = r_hash[0], tau = r_hash[1];
  transcript.append_protocol_name("Lasso MemoryCheckingProof");
  std::vector<fr_t> rand_mem, rand_ops;
  {
    SpanTimer sp(c, "ProductLayer.prove");
    // Subtables::to_grand_products (subtables/mod.rs:133-175) + GrandProducts::new (memory_checking.rs:175-217)
    std::vector<std::unique_ptr<Circuit>> init(alpha), rd(alpha), wr(alpha), fin(alpha);
    DBuf<fr_t> rtree_all(c, G > 1 ? 4 * alpha * 2 * (size_t)G : 0);  // the replicated top layers of every tree
    std::vector<fr_t> rtree_host(G > 1 ? 4 * alpha * 2 * (size_t)G : 0, fr_zero());
    size_t slot = 0;
    for (size_t i = 0; i < alpha; i++) {
      size_t j = (size_t)S.memory_to_dimension_index((int)i), k = (size_t)S.memory_to_subtable_index((int)i);
      for (auto* pc : {&init[i], &fin[i]}) {
        pc->reset(new Circuit());
        circuit_alloc(c, **pc, M, G > 1 ? rtree_all.p + (slot++) * 2 * (size_t)G : nullptr);
      }
      for (auto* pc : {&rd[i], &wr[i]}) {
        pc->reset(new Circuit());
        circuit_alloc(c, **pc, s, G > 1 ? rtree_all.p + (slot++) * 2 * (size_t)G : nullptr);
      }
      launch_gp_fingerprints_mem(tables_fr.p + k * M, dense.fin(j), M_loc, G, gr, gamma, tau, init[i]->tree.p,
                                 fin[i]->tree.p, c->st);
      launch_gp_fingerprints_ops(dense.dim(j), E.p + i * s_loc, dense.read(j), s_loc, gamma, tau, rd[i]->tree.p,
                                 wr[i]->tree.p, c->st);
      g_launches += 2;
    }
    // all trees of a size at once + the top layers straight to the host; without the mapped buffers: tree by tree
    const bool batched = c->h_pub != nullptr;
    std::vector<std::vector<fr_t>> tops(2);  // [0]: init_i, final_i interleaved; [1]: read_i, write_i interleaved
    if (batched) {
      std::vector<std::vector<Circuit*>> groups(2);
      for (size_t i = 0; i < alpha; i++) {
        groups[0].push_back(init[i].get());
        groups[0].push_back(fin[i].get());
        groups[1].push_back(rd[i].get());
        groups[1].push_back(wr[i].get());
      }
      build_trees(c, groups, {M, s}, tops, rtree_host, rtree_all.p);
      if (G > 1)  // pageable source: the copy is staged before the call returns
        LB_CUDA_CHECK(cudaMemcpyAsync(rtree_all.p, rtree_host.data(), rtree_host.size() * sizeof(fr_t), cudaMemcpyHostToDevice, c->st));
    } else {
      if (G > 1) throw std::runtime_error("sharded proof without publication buffers");
      for (size_t i = 0; i < alpha; i++) {
        build_tree(c, *init[i]);
        build_tree(c, *fin[i]);
        build_tree(c, *rd[i]);
        build_tree(c, *wr[i]);
      }
    }
    // ProductLayerProof::prove (memory_checking.rs:673-731)
    transcript.append_protocol_name("Lasso ProductLayerProof");
    auto evaluate = [&](Circuit& ci, int grp, size_t t) {  // grand_product.rs:60-65
      if (batched) return fr_mul(tops[grp][2 * t], tops[grp][2 * t + 1]);
      fr_t top[2];
      c->d2h(top, ci.layer_local(ci.num_layers - 1), 64);
      return fr_mul(top[0], top[1]);
    };
    std::vector<fr_t> claims_rw, claims_if;
    for (size_t i = 0; i < alpha; i++) {
      fr_t hi = evaluate(*init[i], 0, 2 * i), hr = evaluate(*rd[i], 1, 2 * i), hw = evaluate(*wr[i], 1, 2 * i + 1),
           hf = evaluate(*fin[i], 0, 2 * i + 1);
      if (!fr_eq(fr_mul(hi, hw), fr_mul(hr, hf))) throw std::runtime_error("multiset hash check failed (memory_checking.rs:689)");
      transcript.append_scalar("claim_hash_init", hi);
      transcript.append_scalar("claim_hash_read", hr);
      transcript.append_scalar("claim_hash_write", hw);
      transcript.append_scalar("claim_hash_final", hf);
      w.fr(hi);
      w.fr(hr);
      w.fr(hw);
      w.fr(hf);
      claims_rw.push_back(hr);
      claims_rw.push_back(hw);
      claims_if.push_back(hi);
      claims_if.push_back(hf);
    }
    std::vector<Circuit*> rw, inf;
    for (size_t i = 0; i < alpha; i++) {
      rw.push_back(rd[i].get());
      rw.push_back(wr[i].get());
      inf.push_back(init[i].get());
      inf.push_back(fin[i].get());
    }
    GPAProof proof_ops = prove_gpa(c, rw, claims_rw, transcript, rand_ops);
    GPAProof proof_mem = prove_gpa(c, inf, claims_if, transcript, rand_mem);
    ser_gpa(w, proof_mem);  // field order: grand_product_evals, proof_mem, proof_ops (memory_checking.rs:655-660)
    ser_gpa(w, proof_ops);
  }
  {
    // HashLayerProof::prove (memory_checking.rs:337-460)
    SpanTimer sp(c, "HashLayer.prove");
    transcript.append_protocol_name("Lasso HashLayerProof");
    std::vector<fr_t> eval_derefs2(alpha), eval_dim(C), eval_read(C), eval_final(C);
    eq_evals_shard(c, rand_ops, 0, rand_ops.size(), eqtab.p);
    launch_multi_dot_u32(E_u32.p, s_loc, (int)alpha, eqtab.p, s_loc, c->d_partial, c->d_small, c->st);
    launch_multi_dot_u32(dense.d_l_u32.p, s_loc, (int)(2 * C), eqtab.p, s_loc, c->d_partial + 65536, c->d_small + 64, c->st);
    g_launches += 4;
    {
      std::vector<fr_t> tmp(64 + 2 * C);
      reduce_to_host(c, c->d_small, (int)tmp.size(), tmp.data());
      for (size_t i = 0; i < alpha; i++) eval_derefs2[i] = tmp[i];
      for (size_t i = 0; i < C; i++) {
        eval_dim[i] = tmp[64 + i];
        eval_read[i] = tmp[64 + C + i];
      }
    }
    transcript.append_protocol_name("Lasso CombinedTableEvalProof");
    DotProductProofLogBytes proof_derefs =
        prove_joint(c, g, E.p, E_u32.p, nv_d, eval_derefs2, true, "evals_ops_val", "challenge_combine_n_to_one",
                    "joint_claim_eval", rand_ops, transcript, tape);
    eq_evals_shard(c, rand_mem, 0, rand_mem.size(), eqtab.p);
    launch_multi_dot_u32(dense.d_m_u32.p, M_loc, (int)C, eqtab.p, M_loc, c->d_partial, c->d_small, c->st);
    g_launches += 2;
    reduce_to_host(c, c->d_small, (int)C, eval_final.data());
    std::vector<fr_t> evals_ops = eval_dim;
    evals_ops.insert(evals_ops.end(), eval_read.begin(), eval_read.end());
    DotProductProofLogBytes proof_ops =
        prove_joint(c, g, dense.d_l_fr.p, dense.d_l_u32.p, dense.nv_l, evals_ops, true, "claim_evals_ops", "challenge_combine_n_to_one",
                    "joint_claim_eval_ops", rand_ops, transcript, tape);
    // claim_evals_mem is appended UNPADDED and uses Math::log_2 (ceil) of C (memory_checking.rs:413-418)
    DotProductProofLogBytes proof_mem =
        prove_joint(c, g, dense.d_m_fr.p, dense.d_m_u32.p, dense.nv_m, eval_final, false, "claim_evals_mem",
                    "challenge_combine_two_to_one", "joint_claim_eval_mem", rand_mem, transcript, tape);
    // field order (memory_checking.rs:313-329)
    w.arr_fr(eval_dim);
    w.arr_fr(eval_read);
    w.arr_fr(eval_final);
    w.arr_fr(eval_derefs2);
    ser_dpl(w, proof_ops);
    ser_dpl(w, proof_mem);
    ser_dpl(w, proof_derefs);
  }
  c->sync();
  return w.b;
}

}  // namespace lb
