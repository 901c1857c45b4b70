// lasso_b200 — DensifiedRepresentation::from_lookup_indices on the GPU (src/lasso/densified.rs:33-56;
// SURVEY.md §8f-2).  The reference's timestamp loop is sequential per dimension:
//     ts = final[addr]; read[k] = ts; final[addr] = ts + 1
// i.e. read[k] = #{ j < k : addr[j] == addr[k] } and final[a] = #{ k : addr[k] == a }.  Equivalent, and parallel:
// STABLY sort the accesses of a dimension by address; the element at sorted position p (address a, original
// index k) then has read[k] = p - start[a], start = the exclusive scan of the per-address counts (= final).
// The stable sort is an LSD radix sort with 8-bit digits over packed (address << 32 | k) words, all C dimensions
// in the same launches (blockIdx.y = dimension):
//   extract_kernel   column `dim` of the strided index matrix -> packed words (zero-padded to s, densified.rs:33-37),
//                    range check (densified.rs:46), this rank's shard of dim, per-address counts (RED atomics)
//   per 8-bit digit (ceil(log_m / 8) passes):
//     radix_hist_kernel     digit histogram of every tile of 2048 elements -> H[dim][bin][tile]
//     scan_*_kernel         exclusive scan of H in (bin, tile) order = where each tile's run of each digit starts
//     radix_scatter_kernel  every tile IN ORDER, 256 elements per step: rank among equal digits by __match_any_sync
//                           inside the warp + warp-count prefix across the 8 warps + the tile's running count
//   scan_*_kernel    start[a] from the counts; final_ts (this rank's shard) = the counts
//   read_kernel      read[k] = p - start[a] for this rank's k
// Integer, order-preserving, bit-identical to the sequential scan for every input (skew included: nothing here depends
// on how the addresses are distributed).  A few launches of ~10-40 us for 2^20 accesses x 4 dimensions where the host
// scan needs ~3 ms on C threads; no 2^log_m table in shared memory, so any log_m <= 31.
#include <type_traits>

#include "kernels.cuh"

namespace lb {

static constexpr int kRadixThreads = 256;
static constexpr int kRadixRounds = 8;
static constexpr int kRadixTile = kRadixThreads * kRadixRounds;  // 2048 elements per tile
static constexpr uint32_t kDzScanTile = 4096;

// ---------------------------------------------------------------------------------------------- extract
// Element (k, dim) of the n x C index matrix is idx[k * row_stride + dim * col_stride] (element strides >= 0: row-major,
// column-major and broadcast layouts are read in place).  An index that is negative or >= m (densified.rs:46) raises
// *bad (when bad is non-null) and is counted as address 0, so the count atomics below never leave the m counters.
// The host-staged path passes u32 (narrowed and range-checked on the host while staging) with no flag.
template <class T>
__device__ __forceinline__ bool dz_in_range(T v, uint32_t m) {
  if constexpr (std::is_signed<T>::value) return v >= 0 && (uint64_t)v < m;
  else return (uint64_t)v < m;
}
template <class T>
__global__ void __launch_bounds__(256)
    dz_extract_kernel(const T* idx, int64_t row_stride, int64_t col_stride, size_t n, size_t s, uint32_t m, int G, int g,
                      unsigned long long* packed, uint32_t* count, uint32_t* dim_loc_base, size_t dim_stride, uint32_t* bad) {
  const int dim = blockIdx.y;
  const T* col = idx + (int64_t)dim * col_stride;
  unsigned long long* out = packed + (size_t)dim * s;
  uint32_t* cnt = count + (size_t)dim * m;
  uint32_t* dim_loc = dim_loc_base + (size_t)dim * dim_stride;
  for (size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x; k < s; k += (size_t)gridDim.x * blockDim.x) {
    uint32_t a = 0u;
    if (k < n) {
      const T v = col[(int64_t)k * row_stride];
      if (dz_in_range(v, m)) a = (uint32_t)v;
      else if (bad) *bad = 1u;
    }
    out[k] = ((unsigned long long)a << 32) | (unsigned long long)k;
    atomicAdd(cnt + a, 1u);
    if ((int)(k % G) == g) dim_loc[k / G] = a;
  }
}

// ---------------------------------------------------------------------------------------------- radix pass
// H[dim][bin][tile]
__global__ void __launch_bounds__(kRadixThreads)
    dz_radix_hist_kernel(const unsigned long long* in, size_t s, int shift, uint32_t ntiles, uint32_t* H) {
  __shared__ uint32_t h[256];
  const int dim = blockIdx.y;
  const uint32_t tile = blockIdx.x, t = threadIdx.x;
  h[t] = 0;
  __syncthreads();
  const unsigned long long* src = in + (size_t)dim * s + (size_t)tile * kRadixTile;
  const size_t left = s - (size_t)tile * kRadixTile;
#pragma unroll
  for (int r = 0; r < kRadixRounds; r++) {
    const size_t i = (size_t)r * kRadixThreads + t;
    if (i < left) atomicAdd(&h[(uint32_t)(src[i] >> shift) & 0xffu], 1u);
  }
  __syncthreads();
  H[((size_t)dim * 256 + t) * ntiles + tile] = h[t];
}
// stable scatter of one tile; O = exclusive scan of H
__global__ void __launch_bounds__(kRadixThreads)
    dz_radix_scatter_kernel(const unsigned long long* in, unsigned long long* out, size_t s, int shift, uint32_t ntiles,
                            const uint32_t* O) {
  __shared__ uint32_t run[256];    // where the tile's next element of each digit goes
  __shared__ uint32_t wc[8][256];  // per-warp digit counts of the current step
  const int dim = blockIdx.y;
  const uint32_t tile = blockIdx.x, t = threadIdx.x, warp = t >> 5, lane = t & 31;
  run[t] = O[((size_t)dim * 256 + t) * ntiles + tile];
  const unsigned long long* src = in + (size_t)dim * s + (size_t)tile * kRadixTile;
  unsigned long long* dst = out + (size_t)dim * s;
  const size_t left = s - (size_t)tile * kRadixTile;
  for (int r = 0; r < kRadixRounds; r++) {
#pragma unroll
    for (int w = 0; w < 8; w++) wc[w][t] = 0;
    __syncthreads();
    const size_t i = (size_t)r * kRadixThreads + t;
    const bool ok = i < left;
    const unsigned long long e = ok ? src[i] : 0ull;
    // lanes without an element take a value no real digit has (256 + lane): they match nobody
    const uint32_t d = ok ? ((uint32_t)(e >> shift) & 0xffu) : 256u + lane;
    const unsigned peers = __match_any_sync(0xffffffffu, d);
    const uint32_t before = __popc(peers & ((1u << lane) - 1u));
    if (ok && before == 0) wc[warp][d] = (uint32_t)__popc(peers);
    __syncthreads();
    if (ok) {
      uint32_t pos = run[d] + before;
      for (uint32_t w = 0; w < warp; w++) pos += wc[w][d];
      dst[pos] = e;
    }
    __syncthreads();
    uint32_t add = 0;
#pragma unroll
    for (int w = 0; w < 8; w++) add += wc[w][t];
    run[t] += add;
    __syncthreads();
  }
}

// ---------------------------------------------------------------------------------------------- scans
// exclusive scan of `len` counters per dimension (blockIdx.y), in place: tiles of 4096, tile sums, apply
__global__ void __launch_bounds__(1024)
    dz_scan_tiles_kernel(uint32_t* data, size_t len, uint32_t ntiles, uint32_t* tile_sums) {
  __shared__ uint32_t w1[32];
  uint32_t* v = data + (size_t)blockIdx.y * len;
  const uint32_t t = threadIdx.x;
  const size_t base = (size_t)blockIdx.x * kDzScanTile + (size_t)t * 4;
  uint32_t x[4], a = 0;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    x[k] = base + k < len ? v[base + k] : 0u;
    a += x[k];
  }
  uint32_t ia = a;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t ta = __shfl_up_sync(0xffffffffu, ia, d);
    if ((t & 31) >= (uint32_t)d) ia += ta;
  }
  if ((t & 31) == 31) w1[t >> 5] = ia;
  __syncthreads();
  if (t < 32) {
    uint32_t va = w1[t];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t ta = __shfl_up_sync(0xffffffffu, va, d);
      if (t >= (uint32_t)d) va += ta;
    }
    w1[t] = va;
  }
  __syncthreads();
  uint32_t r = ((t >> 5) ? w1[(t >> 5) - 1] : 0u) + ia - a;
#pragma unroll
  for (int k = 0; k < 4; k++) {
    if (base + k < len) v[base + k] = r;
    r += x[k];
  }
  if (t == 1023) tile_sums[(size_t)blockIdx.y * ntiles + blockIdx.x] = w1[31];
}
__global__ void __launch_bounds__(1024) dz_scan_sums_kernel(uint32_t* tile_sums, uint32_t ntiles) {
  __shared__ uint32_t s1[1024];
  uint32_t* ts = tile_sums + (size_t)blockIdx.y * ntiles;
  const uint32_t t = threadIdx.x;
  uint32_t carry = 0;
  for (uint32_t base = 0; base < ntiles; base += 1024) {
    const uint32_t v = base + t < ntiles ? ts[base + t] : 0u;
    s1[t] = v;
    __syncthreads();
    for (uint32_t d = 1; d < 1024; d <<= 1) {
      uint32_t x = 0;
      if (t >= d) x = s1[t - d];
      __syncthreads();
      s1[t] += x;
      __syncthreads();
    }
    if (base + t < ntiles) ts[base + t] = carry + s1[t] - v;
    carry += s1[1023];
    __syncthreads();
  }
}
__global__ void __launch_bounds__(1024)
    dz_scan_apply_kernel(uint32_t* data, size_t len, uint32_t ntiles, const uint32_t* tile_sums) {
  uint32_t* v = data + (size_t)blockIdx.y * len;
  const uint32_t o = tile_sums[(size_t)blockIdx.y * ntiles + blockIdx.x];
  const size_t base = (size_t)blockIdx.x * kDzScanTile + (size_t)threadIdx.x * 4;
#pragma unroll
  for (int k = 0; k < 4; k++)
    if (base + k < len) v[base + k] += o;
}
static int scan_exclusive(uint32_t* data, size_t len, int C, uint32_t* tile_sums, cudaStream_t st) {
  const uint32_t ntiles = (uint32_t)((len + kDzScanTile - 1) / kDzScanTile);
  dim3 grid(ntiles, (unsigned)C);
  dz_scan_tiles_kernel<<<grid, 1024, 0, st>>>(data, len, ntiles, tile_sums);
  LB_LAUNCH_CHECK();
  if (ntiles == 1) return 1;  // a single tile per dimension: its scan is the result
  dz_scan_sums_kernel<<<dim3(1, (unsigned)C), 1024, 0, st>>>(tile_sums, ntiles);
  LB_LAUNCH_CHECK();
  dz_scan_apply_kernel<<<grid, 1024, 0, st>>>(data, len, ntiles, tile_sums);
  LB_LAUNCH_CHECK();
  return 3;
}

// ---------------------------------------------------------------------------------------------- results
// final_ts (this rank's shard: addresses a = i*G + g) = the counts, copied out BEFORE the counts are scanned in place
__global__ void __launch_bounds__(256)
    dz_final_kernel(const uint32_t* count, uint32_t m, int G, int g, uint32_t* final_base, size_t final_stride) {
  const int dim = blockIdx.y;
  const uint32_t a = blockIdx.x * blockDim.x + threadIdx.x;
  if (a >= m) return;
  if ((int)(a % G) == g) final_base[(size_t)dim * final_stride + a / G] = count[(size_t)dim * m + a];
}
// read[k] = p - start[a] (this rank's k: k % G == g, stored at k / G)
__global__ void __launch_bounds__(256)
    dz_read_kernel(const unsigned long long* sorted, size_t s, uint32_t m, const uint32_t* start, int G, int g, uint32_t* read_base,
                   size_t read_stride) {
  const int dim = blockIdx.y;
  const unsigned long long* src = sorted + (size_t)dim * s;
  const uint32_t* st = start + (size_t)dim * m;
  uint32_t* rd = read_base + (size_t)dim * read_stride;
  for (size_t p = (size_t)blockIdx.x * blockDim.x + threadIdx.x; p < s; p += (size_t)gridDim.x * blockDim.x) {
    const unsigned long long e = src[p];
    const uint32_t a = (uint32_t)(e >> 32), k = (uint32_t)e;
    if ((int)(k % G) == g) rd[k / G] = (uint32_t)p - st[a];
  }
}

// function attributes are per device: called from ctx_create for the context's device (nothing to opt into any more)
void densify_init_device() {}
bool densify_gpu_supported(size_t s, size_t log_m) { return log_m >= 1 && log_m <= 31 && s >= 1 && s < ((size_t)1 << 32); }
// scratch (u32 words) for all C dimensions at once
size_t densify_scratch_words(size_t s, int C, size_t log_m) {
  const size_t m = (size_t)1 << log_m;
  const size_t ntiles = (s + kRadixTile - 1) / kRadixTile;
  const size_t H = (size_t)C * 256 * ntiles;
  const size_t scan_len = std::max((size_t)256 * ntiles, m);
  const size_t tsums = (size_t)C * ((scan_len + kDzScanTile - 1) / kDzScanTile + 1);
  return 2 * 2 * (size_t)C * s /* two packed arrays of u64 */ + (size_t)C * m /* counts / start */ + H + tsums + 64;
}
// src: the n x C index matrix on the device.  Outputs are this rank's shards: dim_i at dim_loc + i * dim_stride (likewise
// read, final).  Returns the number of kernels launched.
int launch_densify(const DzSource& src, size_t n, size_t s, int C, size_t log_m, int G, int g, uint32_t* scratch,
                   uint32_t* dim_loc, size_t dim_stride, uint32_t* read_loc, size_t read_stride, uint32_t* final_loc,
                   size_t final_stride, cudaStream_t st) {
  const uint32_t m = 1u << log_m;
  const uint32_t ntiles = (uint32_t)((s + kRadixTile - 1) / kRadixTile);
  unsigned long long* pa = reinterpret_cast<unsigned long long*>(scratch);
  unsigned long long* pb = pa + (size_t)C * s;
  uint32_t* count = reinterpret_cast<uint32_t*>(pb + (size_t)C * s);
  uint32_t* H = count + (size_t)C * m;
  uint32_t* tsums = H + (size_t)C * 256 * ntiles;
  int launches = 0;
  LB_CUDA_CHECK(cudaMemsetAsync(count, 0, (size_t)C * m * 4, st));
  {
    size_t bx = (s + 255) / 256;
    if (bx > (size_t)kNumSMs * 8) bx = kNumSMs * 8;
    const dim3 grid((unsigned)bx, (unsigned)C);
#define LB_DZ_EXTRACT(T)                                                                                                \
  dz_extract_kernel<T><<<grid, 256, 0, st>>>(static_cast<const T*>(src.p), src.row_stride, src.col_stride, n, s, m, G, g, \
                                             pa, count, dim_loc, dim_stride, src.bad)
    switch (src.type) {
      case kDzU64: LB_DZ_EXTRACT(uint64_t); break;
      case kDzI64: LB_DZ_EXTRACT(int64_t); break;
      case kDzU32: LB_DZ_EXTRACT(uint32_t); break;
      case kDzI32: LB_DZ_EXTRACT(int32_t); break;
      default: throw std::runtime_error("launch_densify: unknown index type");
    }
#undef LB_DZ_EXTRACT
    LB_LAUNCH_CHECK();
    launches++;
    if (src.bad_host) {  // the verdict travels to the host while the sort below is already queued
      LB_CUDA_CHECK(cudaMemcpyAsync(src.bad_host, src.bad, 4, cudaMemcpyDeviceToHost, st));
      LB_CUDA_CHECK(cudaEventRecord(src.bad_ready, st));
    }
  }
  unsigned long long *cur = pa, *nxt = pb;
  for (int shift = 0; shift < (int)log_m; shift += 8) {  // LSD: least significant digit first, every pass stable
    dz_radix_hist_kernel<<<dim3(ntiles, (unsigned)C), kRadixThreads, 0, st>>>(cur, s, 32 + shift, ntiles, H);
    LB_LAUNCH_CHECK();
    launches += 1 + scan_exclusive(H, (size_t)256 * ntiles, C, tsums, st);
    dz_radix_scatter_kernel<<<dim3(ntiles, (unsigned)C), kRadixThreads, 0, st>>>(cur, nxt, s, 32 + shift, ntiles, H);
    LB_LAUNCH_CHECK();
    launches++;
    std::swap(cur, nxt);
  }
  dz_final_kernel<<<dim3((m + 255) / 256, (unsigned)C), 256, 0, st>>>(count, m, G, g, final_loc, final_stride);
  LB_LAUNCH_CHECK();
  launches += 1 + scan_exclusive(count, m, C, tsums, st);
  {
    size_t bx = (s + 255) / 256;
    if (bx > (size_t)kNumSMs * 8) bx = kNumSMs * 8;
    dz_read_kernel<<<dim3((unsigned)bx, (unsigned)C), 256, 0, st>>>(cur, s, m, count, G, g, read_loc, read_stride);
    LB_LAUNCH_CHECK();
    launches++;
  }
  return launches;
}

}  // namespace lb
