// libbppgpu: stochastic mapping of event classes on the branches of a tree (Mayrose et al. 2010; the estimator of ChromEvol's
// ComputeChromosomeTransitionsExp).  Semantics in DESIGN.md section 7b.
//
// The generator's off-diagonal is split into T classes, type_rates [T][S][S].  Path n from start state a draws step k from
// Philox4x32-10 (philox.cuh) with key (seed lo, seed hi) and counter (n, a, k, 0):
//   u1 = ((x0 | x1 << 32) >> 11) + 1) 2^-53 in (0, 1]     waiting time -log(u1) / r_i,  r_i = sum_T sum_j type_rates[T][i][j]
//   v  = ((x2 | x3 << 32) >> 11) 2^-53 r_i                event = first (T, j), T-major, j ascending, whose running sum > v
// A state with r_i = 0 is absorbing.  The path runs until its time passes the longest length; a length t reads the state and the
// per-class event counts after every event at time <= t.  One path serves every length.
//
// Tallies are not written per length: between two events the path's record is the same for a run of consecutive lengths in
// increasing order, so the path adds its record at the run's first row of a difference array and subtracts it at the row after
// the run (uint64 arithmetic modulo 2^64), one pair of atomics per class and run, and one prefix pass per (a, j, class) column
// restores the tallies.  Integer sums: the result does not depend on the order of the atomics.
#include "common.cuh"
#include "bppgpu.h"
#include "event_mapping.h"
#include "philox.cuh"
#include "staging.h"

#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

namespace bppgpu {
namespace {

constexpr int kSimThreads = 256;
constexpr size_t kSimSmemMax = 160 * 1024;   // tables above this are read from global memory
thread_local double g_event_ms[2] = {0, 0};

struct SimArgs {
  int S, T, U, nnz;
  const double* len;    // [U] distinct lengths, increasing
  const double* rate;   // [S] r_i
  const double* cum;    // [nnz] running sums of each state's non-zero entries, T-major, j ascending
  const int* off;       // [S + 1] entries of state i: [off[i], off[i + 1])
  const int* code;      // [nnz] class << 16 | target
  uint32_t first;
  unsigned long long n_sims;
  uint32_t k0, k1;
  int use_smem;
  unsigned long long* count;   // [U][S][S] difference array
  unsigned long long* sum;     // [U][S][S][T] difference array
};

// adds the record (state s, class counts c) of path a to the rows [r0, r1) of the difference arrays
__device__ __forceinline__ void add_run(const SimArgs& p, int a, int s, const uint32_t (&c)[kMaxEventTypes], int r0, int r1) {
  const size_t SS = (size_t)p.S * p.S;
  const size_t cell = (size_t)r0 * SS + (size_t)a * p.S + s;
  const size_t step = (size_t)(r1 - r0) * SS;
  atomicAdd(p.count + cell, 1ull);
  if (r1 < p.U) atomicAdd(p.count + cell + step, ~0ull);
#pragma unroll
  for (int t = 0; t < kMaxEventTypes; ++t) {
    if (t < p.T && c[t]) {
      atomicAdd(p.sum + cell * p.T + t, (unsigned long long)c[t]);
      if (r1 < p.U) atomicAdd(p.sum + (cell + step) * p.T + t, 0ull - c[t]);
    }
  }
}

// one thread per path (a, n); a varies fastest, so that a warp's first records go to different cells
__global__ void __launch_bounds__(kSimThreads) event_sim_kernel(SimArgs p) {
  extern __shared__ double sm_tab[];
  if (p.use_smem) {
    double* len = sm_tab;
    double* rate = len + p.U;
    double* cum = rate + p.S;
    int* off = reinterpret_cast<int*>(cum + p.nnz);
    int* code = off + p.S + 1;
    for (int i = threadIdx.x; i < p.U; i += blockDim.x) len[i] = p.len[i];
    for (int i = threadIdx.x; i < p.S; i += blockDim.x) rate[i] = p.rate[i];
    for (int i = threadIdx.x; i < p.nnz; i += blockDim.x) {
      cum[i] = p.cum[i];
      code[i] = p.code[i];
    }
    for (int i = threadIdx.x; i <= p.S; i += blockDim.x) off[i] = p.off[i];
    __syncthreads();
    p.len = len;
    p.rate = rate;
    p.cum = cum;
    p.off = off;
    p.code = code;
  }
  const double tmax = p.len[p.U - 1];
  const unsigned long long total = p.n_sims * (unsigned long long)p.S;
  for (unsigned long long idx = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; idx < total;
       idx += (unsigned long long)gridDim.x * blockDim.x) {
    const int a = (int)(idx % (unsigned)p.S);
    const uint32_t n = p.first + (uint32_t)(idx / (unsigned)p.S);
    uint32_t c[kMaxEventTypes];
#pragma unroll
    for (int t = 0; t < kMaxEventTypes; ++t) c[t] = 0;
    int s = a, row = 0;
    double tau = 0.0;
    for (uint32_t k = 0;; ++k) {
      const double r = p.rate[s];
      if (r == 0.0) break;
      uint32_t x[4] = {n, (uint32_t)a, k, 0u};
      philox4x32_10(x, p.k0, p.k1);
      const unsigned long long h1 = ((unsigned long long)x[0] | (unsigned long long)x[1] << 32) >> 11;
      const unsigned long long h2 = ((unsigned long long)x[2] | (unsigned long long)x[3] << 32) >> 11;
      const double u1 = (double)(h1 + 1) * 0x1p-53;
      tau += -log(u1) / r;
      if (tau > tmax) break;
      // first row whose length is >= tau: rows before it read the record before this event (len[U - 1] = tmax >= tau)
      int lo = row, hi = p.U - 1;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (p.len[mid] < tau) lo = mid + 1;
        else hi = mid;
      }
      if (lo > row) {
        add_run(p, a, s, c, row, lo);
        row = lo;
      }
      const double v = (double)h2 * 0x1p-53 * r;
      int e = p.off[s];
      const int last = p.off[s + 1] - 1;
      while (e < last && !(p.cum[e] > v)) ++e;
      const int cd = p.code[e];
      const int t = cd >> 16;
#pragma unroll
      for (int q = 0; q < kMaxEventTypes; ++q) c[q] += q == t;
      s = cd & 0xFFFF;
    }
    add_run(p, a, s, c, row, p.U);
  }
}

// column col of a [U][X] difference array -> its running sums, in place
__global__ void event_prefix_kernel(unsigned long long* d, int U, long long X) {
  for (long long col = (long long)blockIdx.x * blockDim.x + threadIdx.x; col < X; col += (long long)gridDim.x * blockDim.x) {
    unsigned long long acc = 0;
    for (int u = 0; u < U; ++u) {
      acc += d[(size_t)u * X + col];
      d[(size_t)u * X + col] = acc;
    }
  }
}

// one CTA per branch g of a group: out[t] = sum_{y,x: count > 0} W[x][y] sum[y][x][t] / count[y][x], out[T] = sum_{count = 0}
// W[x][y], where W[x][y] = sum_i w_i joint[i][x][y]; every thread walks fixed cells, then a fixed reduction tree
__global__ void __launch_bounds__(256) event_combine_kernel(const unsigned long long* __restrict__ count,
                                                            const unsigned long long* __restrict__ sum, const int* __restrict__ rows,
                                                            const double* __restrict__ joint, const double* __restrict__ w,
                                                            long long N, int S, int T, const int* __restrict__ out_row,
                                                            double* __restrict__ out) {
  __shared__ double sm[32];
  const int g = blockIdx.x;
  const int SS = S * S;
  count += (size_t)rows[g] * SS;
  sum += (size_t)rows[g] * SS * T;
  joint += (size_t)g * N * SS;
  out += (size_t)out_row[g] * (T + 1);
  double acc[kMaxEventTypes + 1];
#pragma unroll
  for (int q = 0; q <= kMaxEventTypes; ++q) acc[q] = 0.0;
  for (int e = threadIdx.x; e < SS; e += blockDim.x) {
    const int y = e / S, x = e - y * S;
    double W = 0.0;
    for (long long i = 0; i < N; ++i) W += w[i] * joint[((size_t)i * S + x) * S + y];
    const unsigned long long c = count[e];
    if (c) {
      const double dc = (double)c;
#pragma unroll
      for (int q = 0; q < kMaxEventTypes; ++q)
        if (q < T) acc[q] += W * ((double)sum[(size_t)e * T + q] / dc);
    } else {
      acc[kMaxEventTypes] += W;
    }
  }
#pragma unroll
  for (int q = 0; q <= kMaxEventTypes; ++q) {
    if (q < T || q == kMaxEventTypes) {
      const double r = block_sum(acc[q], sm);
      if (threadIdx.x == 0) out[q < T ? q : T] = r;
    }
  }
}

int check_device(int device) {
  int ndev = 0;
  cudaError_t r = cudaGetDeviceCount(&ndev);
  if (r != cudaSuccess || ndev == 0)
    BPP_FAIL(BPPGPU_E_CUDA, "no usable CUDA device (%s); libbppgpu has no CPU fallback", r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
  if (device < 0 || device >= ndev) BPP_FAIL(BPPGPU_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  return BPPGPU_OK;
}

bool on_device(const void* p, int device) {
  cudaPointerAttributes at;
  const bool dev = cudaPointerGetAttributes(&at, p) == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == device;
  cudaGetLastError();
  return dev;
}

}  // namespace

double* event_timing() { return g_event_ms; }

int event_tallies(int device, cudaStream_t st, int S, int T, const double* type_rates, int64_t n_lengths, const double* lengths,
                  int64_t first, int64_t n_sims, uint64_t seed, EventTallies& out, double* ms) {
  if (!type_rates || !lengths) BPP_FAIL(BPPGPU_E_INVALID, "type_rates and lengths must not be NULL");
  if (S < 1 || S > 65535) BPP_FAIL(BPPGPU_E_INVALID, "event mapping takes 1..65535 states, got %d", S);
  if (T < 1 || T > kMaxEventTypes) BPP_FAIL(BPPGPU_E_INVALID, "event mapping takes 1..%d event classes, got %d", kMaxEventTypes, T);
  if (n_lengths < 1 || n_lengths > INT32_MAX) BPP_FAIL(BPPGPU_E_INVALID, "n_lengths must be in 1 .. 2^31 - 1, got %lld", (long long)n_lengths);
  if (n_sims < 1 || first < 0 || first + n_sims > ((int64_t)1 << 32))
    BPP_FAIL(BPPGPU_E_INVALID, "paths %lld .. %lld: need n_sims >= 1 and path indices in 0 .. 2^32 - 1", (long long)first,
             (long long)(first + n_sims - 1));
  const size_t SS = (size_t)S * S;
  std::vector<double> R((size_t)T * SS), len((size_t)n_lengths);
  BPP_CUDA(cudaMemcpy(R.data(), type_rates, R.size() * 8, cudaMemcpyDefault));
  BPP_CUDA(cudaMemcpy(len.data(), lengths, len.size() * 8, cudaMemcpyDefault));
  // per state: its non-zero entries in (class, target) order with their running sums; r_i is the last running sum
  std::vector<int> off(1, 0), code;
  std::vector<double> cum, rate(S);
  for (int i = 0; i < S; ++i) {
    double acc = 0.0;
    for (int t = 0; t < T; ++t)
      for (int j = 0; j < S; ++j) {
        const double v = R[(size_t)t * SS + (size_t)i * S + j];
        if (!std::isfinite(v) || v < 0)
          BPP_FAIL(BPPGPU_E_INVALID, "type_rates[%d][%d][%d] = %g: class rates must be finite and >= 0", t, i, j, v);
        if (i == j && v != 0) BPP_FAIL(BPPGPU_E_INVALID, "type_rates[%d][%d][%d] = %g: the diagonal must be 0", t, i, j, v);
        if (v == 0) continue;
        acc += v;
        cum.push_back(acc);
        code.push_back(t << 16 | j);
      }
    rate[i] = acc;
    off.push_back((int)cum.size());
  }
  for (int64_t b = 0; b < n_lengths; ++b)
    if (!std::isfinite(len[(size_t)b]) || len[(size_t)b] < 0)
      BPP_FAIL(BPPGPU_E_INVALID, "length %lld is %g: lengths must be finite and >= 0", (long long)b, len[(size_t)b]);
  std::vector<double> ulen(len);
  std::sort(ulen.begin(), ulen.end());
  ulen.erase(std::unique(ulen.begin(), ulen.end()), ulen.end());
  const int U = (int)ulen.size();
  out.S = S;
  out.T = T;
  out.U = U;
  out.row_of.resize((size_t)n_lengths);
  for (int64_t b = 0; b < n_lengths; ++b)
    out.row_of[(size_t)b] = (int)(std::lower_bound(ulen.begin(), ulen.end(), len[(size_t)b]) - ulen.begin());

  int rc = check_device(device);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(cudaSetDevice(device));
  const int nnz = (int)cum.size();
  // tables: [len U][rate S][cum nnz] doubles, then [off S + 1][code nnz] ints
  const size_t tab_bytes = ((size_t)U + S + std::max(nnz, 1)) * 8 + ((size_t)S + 1 + std::max(nnz, 1)) * 4;
  std::vector<char> img(tab_bytes, 0);
  double* hd = reinterpret_cast<double*>(img.data());
  std::copy(ulen.begin(), ulen.end(), hd);
  std::copy(rate.begin(), rate.end(), hd + U);
  std::copy(cum.begin(), cum.end(), hd + U + S);
  int* hi = reinterpret_cast<int*>(hd + U + S + std::max(nnz, 1));
  std::copy(off.begin(), off.end(), hi);
  std::copy(code.begin(), code.end(), hi + S + 1);
  void* dtab = nullptr;
  BPP_CUDA(cudaMalloc(&dtab, tab_bytes));
  struct Free { void* p; ~Free() { cudaFree(p); } } free_tab{dtab};
  const size_t bytes_count = (size_t)U * SS * 8, bytes_sum = bytes_count * T;
  BPP_CUDA(cudaMalloc(&out.count, bytes_count));
  BPP_CUDA(cudaMalloc(&out.sum, bytes_sum));
  BPP_CUDA(cudaMemcpyAsync(dtab, img.data(), tab_bytes, cudaMemcpyHostToDevice, st));
  BPP_CUDA(cudaMemsetAsync(out.count, 0, bytes_count, st));
  BPP_CUDA(cudaMemsetAsync(out.sum, 0, bytes_sum, st));

  SimArgs p;
  p.S = S;
  p.T = T;
  p.U = U;
  p.nnz = nnz;
  const double* dd = static_cast<const double*>(dtab);
  p.len = dd;
  p.rate = dd + U;
  p.cum = dd + U + S;
  p.off = reinterpret_cast<const int*>(dd + U + S + std::max(nnz, 1));
  p.code = p.off + S + 1;
  p.first = (uint32_t)first;
  p.n_sims = (unsigned long long)n_sims;
  p.k0 = (uint32_t)seed;
  p.k1 = (uint32_t)(seed >> 32);
  const size_t smem = ((size_t)U + S + nnz) * 8 + ((size_t)S + 1 + nnz) * 4;
  p.use_smem = smem <= kSimSmemMax;
  p.count = out.count;
  p.sum = out.sum;
  const size_t dyn = p.use_smem ? smem : 0;
  if (dyn > 48 * 1024) BPP_CUDA(cudaFuncSetAttribute(event_sim_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
  int sms = 0, occ = 0;
  BPP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device));
  BPP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, event_sim_kernel, kSimThreads, dyn));
  const unsigned long long paths = p.n_sims * (unsigned long long)S;
  // a persistent grid: every CTA copies the tables once
  const unsigned grid = (unsigned)std::max<unsigned long long>(1, std::min<unsigned long long>((paths + kSimThreads - 1) / kSimThreads,
                                                                                               (unsigned long long)std::max(occ, 1) * sms));
  cudaEvent_t ev[2];
  BPP_CUDA(cudaEventCreate(&ev[0]));
  BPP_CUDA(cudaEventCreate(&ev[1]));
  struct EventGuard { cudaEvent_t* e; ~EventGuard() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } evg{ev};
  BPP_CUDA(cudaEventRecord(ev[0], st));
  event_sim_kernel<<<grid, kSimThreads, dyn, st>>>(p);
  BPP_CUDA(cudaGetLastError());
  const long long X[2] = {(long long)SS, (long long)(SS * T)};
  unsigned long long* D[2] = {out.count, out.sum};
  for (int k = 0; k < 2; ++k) {
    event_prefix_kernel<<<(unsigned)std::min<long long>((X[k] + 255) / 256, 65535), 256, 0, st>>>(D[k], U, X[k]);
    BPP_CUDA(cudaGetLastError());
  }
  BPP_CUDA(cudaEventRecord(ev[1], st));
  BPP_CUDA(cudaStreamSynchronize(st));
  float t = 0;
  BPP_CUDA(cudaEventElapsedTime(&t, ev[0], ev[1]));
  if (ms) *ms = t;
  return BPPGPU_OK;
}

cudaError_t event_combine(cudaStream_t st, const EventTallies& t, int n_branches, const int* rows, const double* joint, const double* w,
                          long long N, const int* out_row, double* out) {
  event_combine_kernel<<<n_branches, 256, 0, st>>>(t.count, t.sum, rows, joint, w, N, t.S, t.T, out_row, out);
  return cudaGetLastError();
}

}  // namespace bppgpu

using namespace bppgpu;

int bppgpu_simulate_event_counts(int device, int32_t n_states, int32_t n_types, const double* type_rates, int64_t n_lengths,
                                 const double* lengths, int64_t first_sim, int64_t n_sims, uint64_t seed, uint64_t* count,
                                 uint64_t* sum) {
  if (!count || !sum) BPP_FAIL(BPPGPU_E_INVALID, "count and sum must not be NULL");
  g_event_ms[0] = g_event_ms[1] = 0;
  EventTallies tl;
  cudaStream_t st = nullptr;
  int rc = check_device(device);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(cudaSetDevice(device));
  BPP_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  struct StreamGuard { cudaStream_t s; ~StreamGuard() { cudaStreamDestroy(s); } } sg{st};
  double ms = 0;
  rc = event_tallies(device, st, n_states, n_types, type_rates, n_lengths, lengths, first_sim, n_sims, seed, tl, &ms);
  if (rc != BPPGPU_OK) return rc;
  // length b's rows, in the caller's order; device outputs are written in place, others through the staging pool
  const size_t SS = (size_t)n_states * n_states;
  const size_t rc_bytes = SS * 8, rs_bytes = rc_bytes * n_types;
  const bool dev_c = on_device(count, device), dev_s = on_device(sum, device);
  for (int64_t b = 0; b < n_lengths; ++b) {
    const int r = tl.row_of[(size_t)b];
    void* dc = reinterpret_cast<char*>(count) + (size_t)b * rc_bytes;
    void* ds = reinterpret_cast<char*>(sum) + (size_t)b * rs_bytes;
    const void* sc = tl.count + (size_t)r * SS;
    const void* ss = tl.sum + (size_t)r * SS * n_types;
    if (dev_c) BPP_CUDA(cudaMemcpyAsync(dc, sc, rc_bytes, cudaMemcpyDeviceToDevice, st));
    else BPP_CUDA(staged_copy(dc, sc, rc_bytes, false, device));
    if (dev_s) BPP_CUDA(cudaMemcpyAsync(ds, ss, rs_bytes, cudaMemcpyDeviceToDevice, st));
    else BPP_CUDA(staged_copy(ds, ss, rs_bytes, false, device));
  }
  BPP_CUDA(cudaStreamSynchronize(st));
  g_event_ms[0] = ms;
  return BPPGPU_OK;
}

int bppgpu_expected_events_timing(double* sim_ms, double* combine_ms) {
  if (sim_ms) *sim_ms = g_event_ms[0];
  if (combine_ms) *combine_ms = g_event_ms[1];
  return BPPGPU_OK;
}
