// libbppgpu: site-pattern compression on the device (SURVEY 8f-4, the input side of the hot path).
//
// bpp::SitePatterns::SitePatterns (SitePatterns.cpp:52-106) sorts the alignment columns by their character string and merges
// identical neighbours; bppgpu_site_patterns (engine.cu) is that rule on the host.  Here the same result -- bit for bit: the
// patterns in memcmp order of their columns, each represented by its first site, weights, site -> pattern indices -- is
// produced on the GPU, together with the transposed tip codes the engine consumes, so that a 1M-site x 1024-taxon alignment
// never goes through an O(N log N) string sort on one host core.
//
// Integer / byte work, HBM-bound: nothing here is shaped into a GEMM.
//   1. LSD radix sort of the column permutation, one stable 64-bit pass per 8-byte word of the column from the last word to the
//      first (keys are the word's bytes in big-endian order so that integer order = memcmp order).  The per-pass sort of
//      (key, position) pairs is cub::DeviceRadixSort (a library primitive, like cuBLAS for a plain GEMM); the key gather,
//      run detection, numbering and transposition kernels are below.
//   2. run heads: column[perm[k]] != column[perm[k-1]] (one warp per pair, early exit), inclusive scan -> pattern number.
//   3. scatter: indices[site], pattern_site[pattern] (the run head = smallest original position, the sort being stable),
//      weights[pattern] (integer atomics: order independent).
//   4. tip codes: tip[leaf][pattern] = column[pattern_site[pattern]][leaf] through a shared-memory tile transpose.
#include "common.cuh"
#include "bppgpu.h"
#include "staging.h"

#include <cub/cub.cuh>

#include <algorithm>
#include <chrono>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace bppgpu {

// ---- pageable host memory <-> device at PCIe speed (staging.h) -------------------------------------------------------------------
namespace {
StagePool g_stage;
}  // namespace

cudaError_t StagePool::ensure(int dev) {
  if (device == dev) return cudaSuccess;
  if (device >= 0) return cudaErrorInvalidDevice;   // one device per process for the pool; other devices take the direct copy
  const char* e = getenv("BPPGPU_COPY_THREADS");
  int t = e ? atoi(e) : std::min(4, std::max(1, (int)std::thread::hardware_concurrency()));
  t = std::max(1, std::min(t, kCopyThreadsMax));
  for (int i = 0; i < t; ++i) {
    cudaError_t r = cudaStreamCreateWithFlags(&stream[i], cudaStreamNonBlocking);
    for (int k = 0; k < 2 && r == cudaSuccess; ++k) {
      r = cudaHostAlloc(&pinned[i][k], kStageChunk, cudaHostAllocDefault);
      if (r == cudaSuccess) r = cudaEventCreateWithFlags(&done[i][k], cudaEventDisableTiming);
    }
    if (r != cudaSuccess) return r;
  }
  threads = t;
  device = dev;
  return cudaSuccess;
}

// blocking copy; the caller has synchronised the work that produced `src` (device to host) / will launch consumers afterwards
cudaError_t staged_copy(void* dst, const void* src, size_t bytes, bool h2d, int device) {
  if (bytes == 0) return cudaSuccess;
  const void* host = h2d ? src : dst;
  cudaPointerAttributes at;
  bool pageable = cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeUnregistered;
  cudaGetLastError();
  std::unique_lock<std::mutex> lock(g_stage.mu, std::defer_lock);
  if (pageable && bytes >= 4 * kStageChunk) {
    lock.lock();
    if (g_stage.ensure(device) != cudaSuccess) { cudaGetLastError(); pageable = false; }
  } else {
    pageable = false;
  }
  // (cudaMemcpyDefault: the caller's side may also be DEVICE memory -- an alignment already resident, results that stay on the GPU)
  if (!pageable) return cudaMemcpy(dst, src, bytes, cudaMemcpyDefault);
  const size_t nchunks = (bytes + kStageChunk - 1) / kStageChunk;
  const int T = g_stage.threads;
  std::vector<cudaError_t> err(T, cudaSuccess);
  auto worker = [&](int t) {
    cudaError_t r = cudaSetDevice(device);
    size_t pend_off = 0, pend_len = 0;   // device to host: the chunk whose DMA is in flight, still to be copied out of its slot
    int pend_slot = -1, it = 0;
    for (size_t c = (size_t)t; c < nchunks && r == cudaSuccess; c += (size_t)T, ++it) {
      const int slot = it & 1;
      const size_t off = c * kStageChunk, len = std::min(kStageChunk, bytes - off);
      if (h2d) {
        r = cudaEventSynchronize(g_stage.done[t][slot]);   // the DMA that last read this slot
        if (r != cudaSuccess) break;
        std::memcpy(g_stage.pinned[t][slot], (const char*)src + off, len);
        r = cudaMemcpyAsync((char*)dst + off, g_stage.pinned[t][slot], len, cudaMemcpyHostToDevice, g_stage.stream[t]);
        if (r == cudaSuccess) r = cudaEventRecord(g_stage.done[t][slot], g_stage.stream[t]);
      } else {
        r = cudaMemcpyAsync(g_stage.pinned[t][slot], (const char*)src + off, len, cudaMemcpyDeviceToHost, g_stage.stream[t]);
        if (r == cudaSuccess) r = cudaEventRecord(g_stage.done[t][slot], g_stage.stream[t]);
        if (pend_slot >= 0 && r == cudaSuccess) {
          r = cudaEventSynchronize(g_stage.done[t][pend_slot]);
          if (r == cudaSuccess) std::memcpy((char*)dst + pend_off, g_stage.pinned[t][pend_slot], pend_len);
        }
        pend_slot = slot; pend_off = off; pend_len = len;
      }
    }
    if (r == cudaSuccess) r = cudaStreamSynchronize(g_stage.stream[t]);
    if (!h2d && pend_slot >= 0 && r == cudaSuccess) std::memcpy((char*)dst + pend_off, g_stage.pinned[t][pend_slot], pend_len);
    err[t] = r;
  };
  std::vector<std::thread> th;
  for (int t = 1; t < T; ++t) th.emplace_back(worker, t);
  worker(0);
  for (auto& x : th) x.join();
  for (cudaError_t r : err)
    if (r != cudaSuccess) return r;
  return cudaSuccess;
}

namespace {

// key of position i in this pass: bytes [8w, 8w+8) of column perm[i], first byte most significant, zero padded past the end
__global__ void pattern_key_kernel(const uint8_t* __restrict__ cols, const uint32_t* __restrict__ perm, long long n, int col_bytes,
                                   int word, int aligned8, unsigned long long* __restrict__ keys) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint8_t* c = cols + (size_t)perm[i] * col_bytes + (size_t)word * 8;
  const int rem = col_bytes - word * 8;
  unsigned long long k = 0;
  if (aligned8 && rem >= 8) {
    const unsigned long long v = *reinterpret_cast<const unsigned long long*>(c);   // little-endian load
    const unsigned lo = (unsigned)v, hi = (unsigned)(v >> 32);
    k = ((unsigned long long)__byte_perm(lo, 0, 0x0123) << 32) | (unsigned long long)__byte_perm(hi, 0, 0x0123);
  } else {
    for (int b = 0; b < 8; ++b) k = (k << 8) | (unsigned long long)(b < rem ? c[b] : 0);
  }
  keys[i] = k;
}

__global__ void pattern_iota_kernel(uint32_t* perm, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) perm[i] = (uint32_t)i;
}

// one warp per sorted position k: head[k] = 1 when the column differs from its predecessor (k = 0: always)
__global__ void pattern_head_kernel(const uint8_t* __restrict__ cols, const uint32_t* __restrict__ perm, long long n, int col_bytes,
                                    uint32_t* __restrict__ head) {
  const long long k = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (k >= n) return;
  if (k == 0) {
    if (lane == 0) head[0] = 1u;
    return;
  }
  const uint8_t* a = cols + (size_t)perm[k] * col_bytes;
  const uint8_t* b = cols + (size_t)perm[k - 1] * col_bytes;
  int differ = 0;
  for (int o = 0; o < col_bytes; o += 32) {
    const int j = o + lane;
    const int d = (j < col_bytes) && (a[j] != b[j]);
    if (__any_sync(0xffffffffu, d)) { differ = 1; break; }
  }
  if (lane == 0) head[k] = (uint32_t)differ;
}

// number[k] = inclusive scan of head = 1-based pattern number of sorted position k
__global__ void pattern_scatter_kernel(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ head,
                                       const uint32_t* __restrict__ number, long long n, long long* __restrict__ pattern_site,
                                       uint32_t* __restrict__ weights, long long* __restrict__ indices) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t p = number[k] - 1u;
  const uint32_t site = perm[k];
  indices[site] = (long long)p;
  if (head[k]) pattern_site[p] = (long long)site;
  atomicAdd(&weights[p], 1u);
}

// tip[leaf][pattern] = column[pattern_site[pattern]][leaf], elements of eb bytes; 32 x 32 tiles through shared memory so that
// both the column reads (along the leaf) and the tip-row writes (along the pattern) are contiguous
template <typename T>
__global__ void pattern_tip_codes_kernel(const T* __restrict__ cols, const long long* __restrict__ pattern_site, long long np,
                                         int n_leaves, T* __restrict__ tip) {
  __shared__ T tile[32][33];
  const long long p0 = (long long)blockIdx.x * 32;
  const int l0 = blockIdx.y * 32;
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {   // r = pattern within the tile, threadIdx.x = leaf within the tile
    const long long p = p0 + r;
    const int l = l0 + threadIdx.x;
    if (p < np && l < n_leaves) tile[r][threadIdx.x] = cols[(size_t)pattern_site[p] * n_leaves + l];
  }
  __syncthreads();
  for (int r = threadIdx.y; r < 32; r += blockDim.y) {   // r = leaf within the tile, threadIdx.x = pattern within the tile
    const int l = l0 + r;
    const long long p = p0 + threadIdx.x;
    if (p < np && l < n_leaves) tip[(size_t)l * np + p] = tile[threadIdx.x][r];
  }
}

// ---- "dedup" (the default; BPPGPU_PATTERNS_ALGO=radix selects the plain word-by-word sort of every column) -----------------------
// Measured on 1M sites x 1024 taxa (245k patterns): the kernels of this variant take 20 ms, the plain sort 57 ms; the rest of a call
// is the alignment going in and the tip codes coming out (see staging.h), against 0.59 s for the host routine
// (profiles/r2_patterns_device_vs_host_1Mx1024.json); outputs identical, bit for bit, in every test.
// Identical columns are merged BEFORE the lexicographic sort: one 64-bit hash per column (equal columns -> equal hashes; a
// collision between different columns only leaves duplicates for the final run detection to merge), one stable sort of the hashes,
// run heads by full comparison, and the word-by-word radix sort runs over the unique columns only.
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return x;
}
// one warp per column; position-dependent mixing, commutative combination across lanes
__global__ void pattern_hash_kernel(const uint8_t* __restrict__ cols, long long n, int col_bytes, unsigned long long* __restrict__ hash) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= n) return;
  const uint8_t* c = cols + (size_t)i * col_bytes;
  unsigned long long acc = 0;
  for (int j = lane; j < col_bytes; j += 32) acc += mix64(((unsigned long long)c[j] << 32) ^ (unsigned long long)(j + 1) * 0x9e3779b97f4a7c15ULL);
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) hash[i] = mix64(acc);
}
// sorted by hash: number[k] - 1 = id of the unique column of position k
__global__ void pattern_dedup_scatter_kernel(const uint32_t* __restrict__ perm, const uint32_t* __restrict__ head,
                                             const uint32_t* __restrict__ number, long long n, uint32_t* __restrict__ site_to_u,
                                             uint32_t* __restrict__ u_site, uint32_t* __restrict__ u_weight) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t u = number[k] - 1u, site = perm[k];
  site_to_u[site] = u;
  if (head[k]) u_site[u] = site;     // the run head is the smallest original position: the hash sort is stable
  atomicAdd(&u_weight[u], 1u);
}
// unique columns in lexicographic order: number[k] - 1 = pattern of sorted unique k (several uniques per pattern only after a
// hash collision); pattern_site = smallest original position, weights = summed multiplicities
__global__ void pattern_merge_kernel(const uint32_t* __restrict__ sorted_site, const uint32_t* __restrict__ number, long long nu,
                                     const uint32_t* __restrict__ site_to_u, const uint32_t* __restrict__ u_weight,
                                     long long* __restrict__ pattern_site, uint32_t* __restrict__ weights, uint32_t* __restrict__ u_to_pattern) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= nu) return;
  const uint32_t p = number[k] - 1u, site = sorted_site[k], u = site_to_u[site];
  u_to_pattern[u] = p;
  atomicMin(&pattern_site[p], (long long)site);
  atomicAdd(&weights[p], u_weight[u]);
}
__global__ void pattern_fill_kernel(long long* a, long long n, long long v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) a[i] = v;
}
__global__ void pattern_indices_kernel(const uint32_t* __restrict__ site_to_u, const uint32_t* __restrict__ u_to_pattern, long long n,
                                       long long* __restrict__ indices) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) indices[i] = (long long)u_to_pattern[site_to_u[i]];
}

// every work array comes out of ONE device allocation (a 1M-site call used to pay sixteen cudaMalloc / cudaFree pairs)
struct DevBufs {
  uint8_t* slab = nullptr;
  uint8_t* cols = nullptr;
  unsigned long long *keys_a = nullptr, *keys_b = nullptr;
  uint32_t *perm_a = nullptr, *perm_b = nullptr, *head = nullptr, *number = nullptr, *weights = nullptr;
  long long *pattern_site = nullptr, *indices = nullptr;
  void* temp = nullptr;
  uint8_t* tip = nullptr;
  uint32_t *site_to_u = nullptr, *u_site = nullptr, *u_weight = nullptr, *u_to_pattern = nullptr;   // "dedup" variant
  cudaError_t allocate(long long n, size_t col_total, size_t temp_bytes) {
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += (bytes + 255) & ~(size_t)255; return o; };
    const size_t o_cols = take(col_total + 8);   // + 8: the aligned fast path never reads past the end, the slack is for safety
    const size_t o_ka = take((size_t)n * 8), o_kb = take((size_t)n * 8), o_ps = take((size_t)n * 8), o_ix = take((size_t)n * 8);
    const size_t o_pa = take((size_t)n * 4), o_pb = take((size_t)n * 4), o_hd = take((size_t)n * 4), o_nb = take((size_t)n * 4);
    const size_t o_w = take((size_t)n * 4), o_su = take((size_t)n * 4), o_us = take((size_t)n * 4), o_uw = take((size_t)n * 4);
    const size_t o_up = take((size_t)n * 4), o_tmp = take(std::max<size_t>(temp_bytes, 16));
    const cudaError_t e = cudaMalloc(&slab, off);
    if (e != cudaSuccess) return e;
    cols = slab + o_cols;
    keys_a = reinterpret_cast<unsigned long long*>(slab + o_ka);
    keys_b = reinterpret_cast<unsigned long long*>(slab + o_kb);
    pattern_site = reinterpret_cast<long long*>(slab + o_ps);
    indices = reinterpret_cast<long long*>(slab + o_ix);
    perm_a = reinterpret_cast<uint32_t*>(slab + o_pa);
    perm_b = reinterpret_cast<uint32_t*>(slab + o_pb);
    head = reinterpret_cast<uint32_t*>(slab + o_hd);
    number = reinterpret_cast<uint32_t*>(slab + o_nb);
    weights = reinterpret_cast<uint32_t*>(slab + o_w);
    site_to_u = reinterpret_cast<uint32_t*>(slab + o_su);
    u_site = reinterpret_cast<uint32_t*>(slab + o_us);
    u_weight = reinterpret_cast<uint32_t*>(slab + o_uw);
    u_to_pattern = reinterpret_cast<uint32_t*>(slab + o_up);
    temp = slab + o_tmp;
    return cudaSuccess;
  }
  ~DevBufs() { cudaFree(slab); cudaFree(tip); }
};

// BPPGPU_PATTERNS_TRACE=1: stage times on stderr (each stage synchronised; for profiling, not for timing a production call)
struct StageTrace {
  bool on;
  std::chrono::steady_clock::time_point t0;
  StageTrace() : on(getenv("BPPGPU_PATTERNS_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    cudaDeviceSynchronize();
    const auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[bppgpu patterns] %-28s %8.2f ms\n", what, 1e3 * std::chrono::duration<double>(t1 - t0).count());
    t0 = t1;
  }
};

// The "dedup" variant of steps 1-3 (see above): fills d.pattern_site / d.weights / d.indices and returns the pattern count.
// The buffers of `d` are those the default path allocates; cols are already on the device.
int site_patterns_dedup(DevBufs& d, long long n, int col_bytes, size_t temp_bytes, cudaStream_t st, uint32_t* np_out) {
  const unsigned blocks = (unsigned)((n + 255) / 256);
  const int nwords = (col_bytes + 7) / 8;
  const int aligned8 = col_bytes % 8 == 0;
  auto heads_and_numbers = [&](const uint32_t* perm, long long count, uint32_t* last_number) -> int {
    pattern_head_kernel<<<(unsigned)((count * 32 + 255) / 256), 256, 0, st>>>(d.cols, perm, count, col_bytes, d.head);
    size_t tb = temp_bytes;
    BPP_CUDA(cub::DeviceScan::InclusiveSum(d.temp, tb, d.head, d.number, (int)count, st));
    BPP_CUDA(cudaGetLastError());
    BPP_CUDA(cudaMemcpyAsync(last_number, d.number + (count - 1), 4, cudaMemcpyDeviceToHost, st));
    BPP_CUDA(cudaStreamSynchronize(st));
    return BPPGPU_OK;
  };
  // 1. merge identical columns: hash, stable sort by hash, run heads by full comparison
  pattern_hash_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(d.cols, n, col_bytes, d.keys_a);
  pattern_iota_kernel<<<blocks, 256, 0, st>>>(d.perm_a, n);
  {
    size_t tb = temp_bytes;
    BPP_CUDA(cub::DeviceRadixSort::SortPairs(d.temp, tb, d.keys_a, d.keys_b, d.perm_a, d.perm_b, (int)n, 0, 64, st));
  }
  uint32_t nu32 = 0;
  int rc = heads_and_numbers(d.perm_b, n, &nu32);
  if (rc) return rc;
  const long long nu = (long long)nu32;
  BPP_CUDA(cudaMemsetAsync(d.u_weight, 0, (size_t)n * 4, st));
  pattern_dedup_scatter_kernel<<<blocks, 256, 0, st>>>(d.perm_b, d.head, d.number, n, d.site_to_u, d.u_site, d.u_weight);
  // 2. lexicographic order of the unique columns only: one stable radix pass per 8-byte word, last word first
  BPP_CUDA(cudaMemcpyAsync(d.perm_a, d.u_site, (size_t)nu * 4, cudaMemcpyDeviceToDevice, st));
  uint32_t *pin = d.perm_a, *pout = d.perm_b;
  const unsigned bu = (unsigned)((nu + 255) / 256);
  for (int w = nwords - 1; w >= 0; --w) {
    pattern_key_kernel<<<bu, 256, 0, st>>>(d.cols, pin, nu, col_bytes, w, aligned8, d.keys_a);
    size_t tb = temp_bytes;
    BPP_CUDA(cub::DeviceRadixSort::SortPairs(d.temp, tb, d.keys_a, d.keys_b, pin, pout, (int)nu, 0, 64, st));
    std::swap(pin, pout);
  }
  const uint32_t* sorted = pin;
  rc = heads_and_numbers(sorted, nu, np_out);
  if (rc) return rc;
  // 3. patterns: representative site (smallest original position), weights, site -> pattern
  BPP_CUDA(cudaMemsetAsync(d.weights, 0, (size_t)n * 4, st));
  pattern_fill_kernel<<<bu, 256, 0, st>>>(d.pattern_site, nu, 0x7fffffffffffffffLL);
  pattern_merge_kernel<<<bu, 256, 0, st>>>(sorted, d.number, nu, d.site_to_u, d.u_weight, d.pattern_site, d.weights, d.u_to_pattern);
  pattern_indices_kernel<<<blocks, 256, 0, st>>>(d.site_to_u, d.u_to_pattern, n, d.indices);
  BPP_CUDA(cudaGetLastError());
  BPP_CUDA(cudaStreamSynchronize(st));
  return BPPGPU_OK;
}

// tip codes + copy-out, both variants
int finish_site_patterns(DevBufs& d, long long np, long long n, int col_bytes, int code_bytes, cudaStream_t st, int device,
                         StageTrace& tr, int64_t* pattern_site, uint32_t* weights, int64_t* indices, int64_t* n_patterns, void* tip_codes) {
  if (tip_codes) {
    const int n_leaves = col_bytes / code_bytes;
    BPP_CUDA(cudaMalloc(&d.tip, (size_t)np * (size_t)col_bytes));
    const dim3 grid((unsigned)((np + 31) / 32), (unsigned)((n_leaves + 31) / 32)), block(32, 8);
    if (grid.y > 65535u) BPP_FAIL(BPPGPU_E_INVALID, "too many leaves for the tip-code transpose");
    if (code_bytes == 1)
      pattern_tip_codes_kernel<uint8_t><<<grid, block, 0, st>>>(d.cols, d.pattern_site, np, n_leaves, d.tip);
    else
      pattern_tip_codes_kernel<uint16_t><<<grid, block, 0, st>>>(reinterpret_cast<const uint16_t*>(d.cols), d.pattern_site, np, n_leaves,
                                                                 reinterpret_cast<uint16_t*>(d.tip));
    BPP_CUDA(cudaGetLastError());
  }
  BPP_CUDA(cudaStreamSynchronize(st));
  tr.mark("tip-code transpose");
  BPP_CUDA(staged_copy(pattern_site, d.pattern_site, (size_t)np * 8, false, device));
  BPP_CUDA(staged_copy(weights, d.weights, (size_t)np * 4, false, device));
  BPP_CUDA(staged_copy(indices, d.indices, (size_t)n * 8, false, device));
  if (tip_codes) BPP_CUDA(staged_copy(tip_codes, d.tip, (size_t)np * (size_t)col_bytes, false, device));
  tr.mark("device -> host results");
  *n_patterns = np;
  return BPPGPU_OK;
}

}  // namespace
}  // namespace bppgpu

using namespace bppgpu;

int bppgpu_site_patterns_device(int device, const uint8_t* columns, int64_t n_sites, int32_t col_bytes, int32_t code_bytes,
                                int64_t* pattern_site, uint32_t* weights, int64_t* indices, int64_t* n_patterns,
                                void* tip_codes) {
  if (n_sites < 0 || col_bytes <= 0 || !n_patterns || (n_sites > 0 && (!columns || !pattern_site || !weights || !indices)))
    BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_site_patterns_device");
  if (tip_codes && ((code_bytes != 1 && code_bytes != 2) || col_bytes % code_bytes != 0))
    BPP_FAIL(BPPGPU_E_INVALID, "tip codes need code_bytes 1 or 2 dividing col_bytes");
  if (n_sites >= (int64_t)1 << 31) BPP_FAIL(BPPGPU_E_INVALID, "more than 2^31 - 1 sites");
  int ndev = 0;
  cudaError_t r = cudaGetDeviceCount(&ndev);
  if (r != cudaSuccess || ndev == 0)
    BPP_FAIL(BPPGPU_E_CUDA, "no usable CUDA device (%s); libbppgpu has no CPU fallback", r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
  if (device < 0 || device >= ndev) BPP_FAIL(BPPGPU_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  BPP_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BPP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) BPP_FAIL(BPPGPU_E_CUDA, "device %d is sm_%d%d; libbppgpu is built for sm_100a only", device, prop.major, prop.minor);
  *n_patterns = 0;
  if (n_sites == 0) return BPPGPU_OK;

  const long long n = n_sites;
  const size_t bytes = (size_t)n * (size_t)col_bytes;
  StageTrace tr;
  DevBufs d;
  size_t temp_sort = 0, temp_scan = 0;
  BPP_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, temp_sort, d.keys_a, d.keys_b, d.perm_a, d.perm_b, (int)n));
  BPP_CUDA(cub::DeviceScan::InclusiveSum(nullptr, temp_scan, d.head, d.number, (int)n));
  const size_t temp_bytes = std::max(temp_sort, temp_scan);
  BPP_CUDA(d.allocate(n, bytes, temp_bytes));
  tr.mark("device allocation");

  cudaStream_t st = 0;
  BPP_CUDA(staged_copy(d.cols, columns, bytes, true, device));
  tr.mark("host -> device alignment");
  const char* algo = getenv("BPPGPU_PATTERNS_ALGO");
  if (!(algo && std::string(algo) == "radix")) {
    uint32_t npd = 0;
    const int rc = site_patterns_dedup(d, n, col_bytes, temp_bytes, st, &npd);
    if (rc) return rc;
    tr.mark("dedup + sort + numbering");
    return finish_site_patterns(d, (long long)npd, n, col_bytes, code_bytes, st, device, tr, pattern_site, weights, indices, n_patterns, tip_codes);
  }
  const unsigned blocks = (unsigned)((n + 255) / 256);
  pattern_iota_kernel<<<blocks, 256, 0, st>>>(d.perm_a, n);
  const int nwords = (col_bytes + 7) / 8;
  const int aligned8 = col_bytes % 8 == 0;
  uint32_t *pin = d.perm_a, *pout = d.perm_b;
  for (int w = nwords - 1; w >= 0; --w) {
    pattern_key_kernel<<<blocks, 256, 0, st>>>(d.cols, pin, n, col_bytes, w, aligned8, d.keys_a);
    size_t tb = temp_bytes;
    BPP_CUDA(cub::DeviceRadixSort::SortPairs(d.temp, tb, d.keys_a, d.keys_b, pin, pout, (int)n, 0, 64, st));
    std::swap(pin, pout);
  }
  const uint32_t* perm = pin;   // sorted positions -> original site
  pattern_head_kernel<<<(unsigned)((n * 32 + 255) / 256), 256, 0, st>>>(d.cols, perm, n, col_bytes, d.head);
  {
    size_t tb = temp_bytes;
    BPP_CUDA(cub::DeviceScan::InclusiveSum(d.temp, tb, d.head, d.number, (int)n, st));
  }
  BPP_CUDA(cudaMemsetAsync(d.weights, 0, (size_t)n * 4, st));
  pattern_scatter_kernel<<<blocks, 256, 0, st>>>(perm, d.head, d.number, n, d.pattern_site, d.weights, d.indices);
  BPP_CUDA(cudaGetLastError());
  uint32_t np32 = 0;
  BPP_CUDA(cudaMemcpyAsync(&np32, d.number + (n - 1), 4, cudaMemcpyDeviceToHost, st));
  BPP_CUDA(cudaStreamSynchronize(st));
  tr.mark("radix sort + numbering");
  return finish_site_patterns(d, (long long)np32, n, col_bytes, code_bytes, st, device, tr, pattern_site, weights, indices, n_patterns, tip_codes);
}
