// libbppgpu: pairwise maximum-likelihood distances (DistanceEstimation::computeMatrix, Distance/DistanceEstimation.cpp, with
// one TwoTreeLikelihood per pair of sequences).  Semantics in DESIGN.md section 7b.
//
// The per-pair sufficient statistic is the table of joint code counts n_ab[u][v] = sum_k w_k [code_a(k) = u][code_b(k) = v].
// All of them together are one integer matrix product n = E diag(w) E^T over the patterns, E the one-hot matrix
// [(leaf, code)][pattern]:
//   1. pack: tip codes -> one uint8 row per leaf, padded to a multiple of kChunk patterns.  A pattern of weight w > 127 becomes
//      ceil(w / 127) virtual columns of weight <= 127 each, so that every weight fits a signed 8-bit operand.
//   2. counts: mma.sync m16n8k32 s8 x s8 -> s32 (IMMA).  The operand fragments are built in registers straight from the code
//      bytes (__vcmpeq4 against the row's / column's code; the B side ANDed with the weight bytes): E is never materialised.
//      Only 128 x 128 tiles on or above the diagonal run; pattern slices add their integer tiles into the count buffer with
//      integer atomics, so counts are exact and identical from run to run.  Above kCountBudget bytes of counts, the pairs are
//      processed in blocks of consecutive first leaves.
//   3. ML: a warp per pair maximises lnL_ab(t) = sum_uv n_ab[u][v] log f_uv(t) on [1e-6, 1e4] in the spectral form
//      f_uv(t) = sum_j A[u][j] B[v][j] g_j(t), g_j(t) = sum_c p_c exp(lambda_j rho r_c t), with a fixed search: a 64-point log grid,
//      the bracket of the best grid point, then safeguarded Newton / log-bisection on d lnL / dt.
#include "common.cuh"
#include "bppgpu.h"
#include "staging.h"

#include <algorithm>
#include <cmath>
#include <cstring>
#include <vector>

namespace bppgpu {
namespace {

constexpr int kMaxCodes = 128;                    // codes are compared as signed-8-bit-safe bytes
constexpr int kChunk = 128;                       // patterns per shared-memory stage of the count kernel
constexpr int kRowStride = kChunk + 16;           // bytes per leaf row in shared memory: fragment loads hit distinct banks
constexpr int kTile = 128;                        // (leaf, code) rows and columns per count CTA
constexpr int kTileLeaves = kTile + 1;            // leaves a tile side can touch: floor(127 / K) + 2
constexpr size_t kCountBudget = (size_t)512 << 20;   // device bytes of pair counts held at once
constexpr int kGrid = 64;                         // log-spaced probes of the ML search
constexpr int kMaxNewton = 100;
constexpr double kTmin = 1e-6, kTmax = 1e4;       // TwoTreeLikelihood's branch-length bounds
constexpr int kMlWarps = 4;

struct DevMem {
  void* p = nullptr;
  ~DevMem() { cudaFree(p); }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// out[l][j] = code of virtual column j of leaf l (0 with weight 0 in the padding); codes >= n_codes raise *bad
template <typename T>
__global__ void dist_pack_kernel(const T* __restrict__ codes, long long n, const uint32_t* __restrict__ vcol, long long nv,
                                 long long npad, int n_codes, uint8_t* __restrict__ out, int* __restrict__ bad) {
  const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int l = blockIdx.y;
  if (j >= npad) return;
  uint8_t c = 0;
  if (j < nv) {
    const unsigned v = codes[(size_t)l * n + (vcol ? vcol[j] : j)];
    if (v >= (unsigned)n_codes) atomicOr(bad, 1);
    else c = (uint8_t)v;
  }
  out[(size_t)l * npad + j] = c;
}

__device__ __forceinline__ void imma16832(int* c, const unsigned* a, const unsigned* b) {
  asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.s8.s8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}

__host__ __device__ __forceinline__ long long pair_index(long long a, long long b, long long L) {
  return a * (2 * L - a - 1) / 2 + (b - a - 1);
}

// One CTA: rows [r0, r0 + 128) x columns [c0, c0 + 128) of n = E diag(w) E^T (row / column index = leaf * K + code) over the
// kChunk-pattern chunks of slice blockIdx.z.  8 warps as 2 x 4, each 64 x 32 = 4 x 4 m16n8 tiles.  Entries of pairs a < b with
// a in [a0, a1) are added into counts[(pair - pair_base)][u][v].
__global__ void __launch_bounds__(256) dist_count_kernel(const uint8_t* __restrict__ codes, const uint8_t* __restrict__ w8,
                                                         long long npad, int L, int K, int ti0, int a0, int a1, long long pair_base,
                                                         long long chunks_per_slice, unsigned* __restrict__ counts) {
  const int ti = ti0 + blockIdx.y, tj = blockIdx.x;
  if (tj < ti) return;
  __shared__ __align__(16) uint8_t sA[kTileLeaves * kRowStride];
  __shared__ __align__(16) uint8_t sB[kTileLeaves * kRowStride];
  __shared__ __align__(16) uint8_t sW[kChunk];
  const int rows = L * K;
  const int r0 = ti * kTile, c0 = tj * kTile;
  const int la0 = r0 / K, lb0 = c0 / K;
  const int nA = (min(r0 + kTile, rows) - 1) / K - la0 + 1;   // leaves the tile's rows touch
  const int nB = (min(c0 + kTile, rows) - 1) / K - lb0 + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, tig = lane & 3;
  const int wm = warp >> 2, wn = warp & 3;
  // the (leaf, code) of every fragment row / column this thread reads; rows past the end never match (codes are < 128)
  int aoff[8], boff[4];
  unsigned arep[8], brep[4];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int R = r0 + wm * 64 + (i >> 1) * 16 + g + (i & 1) * 8;
    aoff[i] = R < rows ? (R / K - la0) * kRowStride : 0;
    arep[i] = R < rows ? (unsigned)(R % K) * 0x01010101u : 0xffffffffu;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int Cc = c0 + wn * 32 + i * 8 + g;
    boff[i] = Cc < rows ? (Cc / K - lb0) * kRowStride : 0;
    brep[i] = Cc < rows ? (unsigned)(Cc % K) * 0x01010101u : 0xffffffffu;
  }
  int acc[4][4][4];
#pragma unroll
  for (int m = 0; m < 4; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int q = 0; q < 4; ++q) acc[m][n][q] = 0;

  const long long nchunks = npad / kChunk;
  const long long kc0 = (long long)blockIdx.z * chunks_per_slice, kc1 = min(nchunks, kc0 + chunks_per_slice);
  const int nload = (nA + nB) * (kChunk / 16) + kChunk / 16;
  for (long long kc = kc0; kc < kc1; ++kc) {
    const long long p0 = kc * kChunk;
    __syncthreads();
    for (int i = threadIdx.x; i < nload; i += blockDim.x) {
      const int row = i / (kChunk / 16), part = i % (kChunk / 16);
      const uint8_t* src;
      uint8_t* dst;
      if (row < nA) { src = codes + (size_t)(la0 + row) * npad; dst = sA + row * kRowStride; }
      else if (row < nA + nB) { src = codes + (size_t)(lb0 + row - nA) * npad; dst = sB + (row - nA) * kRowStride; }
      else { src = w8; dst = sW; }
      *reinterpret_cast<uint4*>(dst + part * 16) = __ldg(reinterpret_cast<const uint4*>(src + p0 + part * 16));
    }
    __syncthreads();
#pragma unroll
    for (int ks = 0; ks < kChunk; ks += 32) {
      const int k = ks + tig * 4;
      const unsigned w0 = *reinterpret_cast<const unsigned*>(sW + k), w1 = *reinterpret_cast<const unsigned*>(sW + k + 16);
      unsigned a[4][4], b[4][2];
#pragma unroll
      for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint8_t* s = sA + aoff[m * 2 + h] + k;
          a[m][h] = __vcmpeq4(*reinterpret_cast<const unsigned*>(s), arep[m * 2 + h]) & 0x01010101u;
          a[m][2 + h] = __vcmpeq4(*reinterpret_cast<const unsigned*>(s + 16), arep[m * 2 + h]) & 0x01010101u;
        }
#pragma unroll
      for (int n = 0; n < 4; ++n) {
        const uint8_t* s = sB + boff[n] + k;
        b[n][0] = __vcmpeq4(*reinterpret_cast<const unsigned*>(s), brep[n]) & w0;
        b[n][1] = __vcmpeq4(*reinterpret_cast<const unsigned*>(s + 16), brep[n]) & w1;
      }
#pragma unroll
      for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int n = 0; n < 4; ++n) imma16832(acc[m][n], a[m], b[n]);
    }
  }
#pragma unroll
  for (int m = 0; m < 4; ++m)
#pragma unroll
    for (int n = 0; n < 4; ++n)
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int v = acc[m][n][q];
        const int R = r0 + wm * 64 + m * 16 + g + (q >> 1) * 8, Cc = c0 + wn * 32 + n * 8 + tig * 2 + (q & 1);
        if (v == 0 || R >= rows || Cc >= rows) continue;
        const int ra = R / K, cb = Cc / K;
        if (ra < a0 || ra >= a1 || cb <= ra) continue;
        const long long p = pair_index(ra, cb, L) - pair_base;
        atomicAdd(&counts[(size_t)p * K * K + (size_t)(R % K) * K + (Cc % K)], (unsigned)v);
      }
}

struct MlArgs {
  const unsigned* counts;   // [npairs][K][K]
  long long npairs;
  int K, S, C;
  const double* A;          // [K][S]  sum_x pi_x e_u(x) V[x][j]
  const double* B;          // [K][S]  sum_y V^-1[j][y] e_v(y)
  const double* mu;         // [S]     lambda_j * rho
  const double* rates;      // [C]
  const double* probs;      // [C]
  const uint8_t* ambiguous; // [K]     code row is all ones: f_uv does not depend on t
  double* dist;             // [npairs]
  double* lnl;              // [npairs]
};

struct Probe {
  double l, d1, d2;
  bool bad;   // some informative cell had f_uv(t) <= 0: lnL = -inf there
};

// lnL and its first two t-derivatives at t for the pair whose counts are `cnt`; every lane of the warp calls it.  Cells are summed
// per lane in a fixed order, then across lanes by a fixed shuffle tree: the result does not depend on timing.
__device__ Probe ml_probe(const MlArgs& a, const unsigned* __restrict__ cnt, double t, double* g, int lane) {
  const int S = a.S, KK = a.K * a.K;
  __syncwarp();
  for (int j = lane; j < S; j += 32) {
    double g0 = 0, g1 = 0, g2 = 0;
    for (int c = 0; c < a.C; ++c) {
      const double x = a.mu[j] * a.rates[c], e = a.probs[c] * exp(x * t);
      g0 += e;
      g1 += x * e;
      g2 += x * x * e;
    }
    g[j] = g0;
    g[S + j] = g1;
    g[2 * S + j] = g2;
  }
  __syncwarp();
  double l = 0, d1 = 0, d2 = 0;
  bool bad = false;
  for (int idx = lane; idx < KK; idx += 32) {
    const unsigned n = cnt[idx];
    if (n == 0) continue;
    const double* Au = a.A + (size_t)(idx / a.K) * S;
    const double* Bv = a.B + (size_t)(idx % a.K) * S;
    double f = 0, f1 = 0, f2 = 0;
    for (int j = 0; j < S; ++j) {
      const double ab = Au[j] * Bv[j];
      f += ab * g[j];
      f1 += ab * g[S + j];
      f2 += ab * g[2 * S + j];
    }
    if (!(f > 0)) { bad = true; continue; }
    const double r1 = f1 / f;
    l += n * log(f);
    d1 += n * r1;
    d2 += n * (f2 / f - r1 * r1);
  }
  Probe p;
  p.l = warp_sum(l);
  p.d1 = warp_sum(d1);
  p.d2 = warp_sum(d2);
  p.bad = __any_sync(0xffffffffu, bad);
  return p;
}

__device__ __forceinline__ double grid_t(int i) {
  if (i == 0) return kTmin;
  if (i == kGrid - 1) return kTmax;
  return exp(log(kTmin) + (log(kTmax) - log(kTmin)) * i / (kGrid - 1));
}

// one warp per pair
__global__ void __launch_bounds__(kMlWarps * 32) dist_ml_kernel(MlArgs a) {
  extern __shared__ double smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long p = (long long)blockIdx.x * kMlWarps + warp;
  if (p >= a.npairs) return;
  double* g = smem + (size_t)warp * 3 * a.S;
  const unsigned* cnt = a.counts + (size_t)p * a.K * a.K;
  // a pair with no informative cell (each involves a fully ambiguous code) is flat: the reference's start value 1e-6
  bool informative = false;
  for (int idx = lane; idx < a.K * a.K; idx += 32)
    if (cnt[idx] && !a.ambiguous[idx / a.K] && !a.ambiguous[idx % a.K]) informative = true;
  double t = kTmin;
  Probe best = ml_probe(a, cnt, kTmin, g, lane);
  if (__any_sync(0xffffffffu, informative)) {
    // 1. grid; ties go to the larger t (a plateau reached in floating point at large t is the upper bound's value)
    int ib = 0;
    for (int i = 1; i < kGrid; ++i) {
      const Probe q = ml_probe(a, cnt, grid_t(i), g, lane);
      if (!q.bad && (best.bad || q.l >= best.l)) { best = q; ib = i; }
    }
    t = grid_t(ib);
    // 2. bracket from the sign of d lnL / dt at the best probe.  No search: the optimum is on the bound the slope points to
    //    (returned exactly), d lnL / dt vanishes at the probe, or every probe was -inf (a code row of zeros)
    double lo = 0, hi = 0;
    bool search = false;
    if (!best.bad && best.d1 > 0 && ib < kGrid - 1) { search = true; lo = t; hi = grid_t(ib + 1); }
    else if (!best.bad && best.d1 < 0 && ib > 0) { search = true; lo = grid_t(ib - 1); hi = t; }
    // 3. safeguarded Newton on d lnL / dt, log-bisection when the Newton step leaves the bracket or lnL is not concave there
    if (search) {
      Probe cur = best;
      double tc = t;
      for (int it = 0; it < kMaxNewton; ++it) {
        double tn = (!cur.bad && cur.d2 < 0) ? tc - cur.d1 / cur.d2 : -1.0;
        if (!(tn > lo && tn < hi)) tn = sqrt(lo * hi);
        const double step = fabs(tn - tc);
        tc = tn;
        cur = ml_probe(a, cnt, tc, g, lane);
        if (cur.bad || cur.d1 > 0) lo = tc;   // f <= 0 only happens below the optimum (t -> 0 cancellation)
        else if (cur.d1 < 0) hi = tc;
        if ((!cur.bad && cur.d1 == 0) || step <= 1e-12 * tc) break;
      }
      // (a guard for lnL with several local maxima in the bracket; at a converged optimum the values agree to rounding)
      if (!cur.bad && cur.l >= best.l - 1e-12 * fabs(best.l)) { best = cur; t = tc; }
    }
  }
  if (lane == 0) {
    a.dist[p] = t;
    a.lnl[p] = best.bad ? -INFINITY : best.l;
  }
}

// Pattern slices per count tile: every (tile, slice) CTA does the same work, so the count launch takes ceil(tiles * slices / slots)
// waves of `slots` resident CTAs.  The fewest slices that fill the card and keep the last wave at least 95 % full (else the best
// fill up to 32 slices): at 1024 taxa x 4 codes, 528 tiles on 2 x 148 slots, 2 slices leave the fourth wave 57 % full, 5 fill nine
// waves to 99 %.
long long count_slices(long long tiles, long long nchunks, long long slots) {
  long long best = 1;
  double best_fill = 0;
  for (long long s = 1; s <= std::min<long long>(nchunks, 32); ++s) {
    const long long ctas = tiles * s, waves = (ctas + slots - 1) / slots;
    const double fill = (double)ctas / (double)(waves * slots);
    if (ctas >= slots && fill >= 0.95) return s;
    if (fill > best_fill + 1e-9) { best_fill = fill; best = s; }
  }
  return best;
}

thread_local double g_last_ms[3] = {0, 0, 0};

}  // namespace
}  // namespace bppgpu

using namespace bppgpu;

int bppgpu_pairwise_distances(int device, const bppgpu_model_desc* model, const double* freqs, int32_t n_cats, const double* rates,
                              const double* probs, int32_t n_codes, int32_t code_bytes, const double* code_table, int32_t n_leaves,
                              int64_t n_patterns, const void* tip_codes, const uint32_t* weights, double* dist, double* lnl,
                              uint32_t* counts) {
  if (!model || !freqs || !rates || !probs || !code_table || !tip_codes || !weights || !dist || n_cats < 1 || n_patterns < 1)
    BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_pairwise_distances");
  if (n_leaves < 2 || n_leaves > 65535) BPP_FAIL(BPPGPU_E_INVALID, "pairwise distances need 2..65535 sequences, got %d", n_leaves);
  if (n_codes < 1 || n_codes > kMaxCodes) BPP_FAIL(BPPGPU_E_INVALID, "pairwise distances take 1..%d tip codes, got %d", kMaxCodes, n_codes);
  if (code_bytes != 1 && code_bytes != 2) BPP_FAIL(BPPGPU_E_INVALID, "code_bytes must be 1 or 2");
  const int S = model->n_states;
  const unsigned need = BPPGPU_MODEL_DIAGONALIZABLE | BPPGPU_MODEL_NONSINGULAR;
  if (S < 1 || !model->right_eigen || !model->left_eigen || !model->eigen_re || (model->flags & need) != need ||
      (model->flags & (BPPGPU_MODEL_CLAMP01 | BPPGPU_MODEL_CHR_TAYLOR)))
    BPP_FAIL(BPPGPU_E_INVALID, "pairwise distances need a diagonalizable, non-singular model with the plain eigen form of P(t)");
  if (model->eigen_im)
    for (int j = 0; j < S; ++j)
      if (model->eigen_im[j] != 0) BPP_FAIL(BPPGPU_E_INVALID, "pairwise distances need a real spectrum (eigenvalue %d is complex)", j);
  int ndev = 0;
  cudaError_t r = cudaGetDeviceCount(&ndev);
  if (r != cudaSuccess || ndev == 0)
    BPP_FAIL(BPPGPU_E_CUDA, "no usable CUDA device (%s); libbppgpu has no CPU fallback", r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
  if (device < 0 || device >= ndev) BPP_FAIL(BPPGPU_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  BPP_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BPP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) BPP_FAIL(BPPGPU_E_CUDA, "device %d is sm_%d%d; libbppgpu is built for sm_100a only", device, prop.major, prop.minor);

  const long long L = n_leaves, N = n_patterns;
  const int K = n_codes;
  cudaStream_t st = 0;
  cudaEvent_t ev[2];
  BPP_CUDA(cudaEventCreate(&ev[0]));
  BPP_CUDA(cudaEventCreate(&ev[1]));
  struct EventGuard { cudaEvent_t* e; ~EventGuard() { cudaEventDestroy(e[0]); cudaEventDestroy(e[1]); } } evg{ev};
  auto elapsed = [&](float& ms) { cudaEventSynchronize(ev[1]); return cudaEventElapsedTime(&ms, ev[0], ev[1]); };
  double ms_upload = 0, ms_count = 0, ms_ml = 0;
  float ms = 0;

  // ---- 1. weights -> virtual columns of weight <= 127 ---------------------------------------------------------------------
  BPP_CUDA(cudaEventRecord(ev[0], st));
  std::vector<uint32_t> w((size_t)N);
  BPP_CUDA(cudaMemcpy(w.data(), weights, (size_t)N * 4, cudaMemcpyDefault));
  unsigned long long total = 0;
  long long nv = 0;
  bool split = false;   // virtual column j is pattern j only when every weight is in [1, 127]
  for (uint32_t x : w) {
    total += x;
    nv += (x + 126) / 127;
    split = split || x == 0 || x > 127;
  }
  if (total >= (1ull << 31)) BPP_FAIL(BPPGPU_E_INVALID, "total pattern weight %llu does not fit the int32 counts (must be < 2^31)", total);
  const long long npad = std::max<long long>(kChunk, (nv + kChunk - 1) / kChunk * kChunk);
  std::vector<uint8_t> w8((size_t)npad, 0);
  std::vector<uint32_t> vcol(split ? (size_t)nv : 0);
  for (long long k = 0, j = 0; k < N; ++k)
    for (uint32_t left = w[(size_t)k]; left > 0; ++j) {
      const uint32_t take = std::min<uint32_t>(left, 127);
      w8[(size_t)j] = (uint8_t)take;
      if (split) vcol[(size_t)j] = (uint32_t)k;
      left -= take;
    }

  // ---- 2. tip codes on the device (read in place when they already are), packed to uint8 rows -------------------------------
  const size_t code_total = (size_t)L * (size_t)N * (size_t)code_bytes;
  cudaPointerAttributes at;
  const bool resident = cudaPointerGetAttributes(&at, tip_codes) == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == device;
  cudaGetLastError();
  DevMem raw, packed, dw8, dvcol, dbad;
  const void* src = tip_codes;
  if (!resident) {
    BPP_CUDA(cudaMalloc(&raw.p, code_total));
    BPP_CUDA(staged_copy(raw.p, tip_codes, code_total, true, device));
    src = raw.p;
  }
  BPP_CUDA(cudaMalloc(&packed.p, (size_t)L * (size_t)npad));
  BPP_CUDA(cudaMalloc(&dw8.p, (size_t)npad));
  BPP_CUDA(cudaMalloc(&dbad.p, 4));
  BPP_CUDA(cudaMemcpyAsync(dw8.p, w8.data(), (size_t)npad, cudaMemcpyHostToDevice, st));
  BPP_CUDA(cudaMemsetAsync(dbad.p, 0, 4, st));
  if (split) {
    BPP_CUDA(cudaMalloc(&dvcol.p, (size_t)nv * 4));
    BPP_CUDA(cudaMemcpyAsync(dvcol.p, vcol.data(), (size_t)nv * 4, cudaMemcpyHostToDevice, st));
  }
  {
    const dim3 grid((unsigned)((npad + 255) / 256), (unsigned)L);
    if (code_bytes == 1)
      dist_pack_kernel<uint8_t><<<grid, 256, 0, st>>>(static_cast<const uint8_t*>(src), N, dvcol.as<uint32_t>(), nv, npad, K,
                                                      packed.as<uint8_t>(), dbad.as<int>());
    else
      dist_pack_kernel<uint16_t><<<grid, 256, 0, st>>>(static_cast<const uint16_t*>(src), N, dvcol.as<uint32_t>(), nv, npad, K,
                                                       packed.as<uint8_t>(), dbad.as<int>());
    BPP_CUDA(cudaGetLastError());
  }
  int bad = 0;
  BPP_CUDA(cudaMemcpyAsync(&bad, dbad.p, 4, cudaMemcpyDeviceToHost, st));
  BPP_CUDA(cudaEventRecord(ev[1], st));
  BPP_CUDA(cudaStreamSynchronize(st));
  if (bad) BPP_FAIL(BPPGPU_E_INVALID, "a tip code is >= n_codes (%d)", K);
  BPP_CUDA(elapsed(ms));
  ms_upload = ms;
  cudaFree(raw.p);   // the packed rows are all the kernels read
  raw.p = nullptr;

  // ---- 3. spectral coefficients (host, FP64) --------------------------------------------------------------------------------
  std::vector<double> A((size_t)K * S, 0.0), Bm((size_t)K * S, 0.0), mu(S);
  std::vector<uint8_t> amb(K);
  for (int u = 0; u < K; ++u) {
    const double* e = code_table + (size_t)u * S;
    bool all = true;
    for (int x = 0; x < S; ++x) all = all && e[x] == 1.0;
    amb[u] = all;
    for (int j = 0; j < S; ++j) {
      double sa = 0, sb = 0;
      for (int x = 0; x < S; ++x) {
        sa += freqs[x] * e[x] * model->right_eigen[(size_t)x * S + j];
        sb += model->left_eigen[(size_t)j * S + x] * e[x];
      }
      A[(size_t)u * S + j] = sa;
      Bm[(size_t)u * S + j] = sb;
    }
  }
  for (int j = 0; j < S; ++j) mu[j] = model->eigen_re[j] * model->rate;
  DevMem dA, dB, dmu, drt, dpr, damb;
  BPP_CUDA(cudaMalloc(&dA.p, A.size() * 8));
  BPP_CUDA(cudaMalloc(&dB.p, Bm.size() * 8));
  BPP_CUDA(cudaMalloc(&dmu.p, (size_t)S * 8));
  BPP_CUDA(cudaMalloc(&drt.p, (size_t)n_cats * 8));
  BPP_CUDA(cudaMalloc(&dpr.p, (size_t)n_cats * 8));
  BPP_CUDA(cudaMalloc(&damb.p, (size_t)K));
  BPP_CUDA(cudaMemcpy(dA.p, A.data(), A.size() * 8, cudaMemcpyHostToDevice));
  BPP_CUDA(cudaMemcpy(dB.p, Bm.data(), Bm.size() * 8, cudaMemcpyHostToDevice));
  BPP_CUDA(cudaMemcpy(dmu.p, mu.data(), (size_t)S * 8, cudaMemcpyHostToDevice));
  BPP_CUDA(cudaMemcpy(drt.p, rates, (size_t)n_cats * 8, cudaMemcpyDefault));
  BPP_CUDA(cudaMemcpy(dpr.p, probs, (size_t)n_cats * 8, cudaMemcpyDefault));
  BPP_CUDA(cudaMemcpy(damb.p, amb.data(), (size_t)K, cudaMemcpyHostToDevice));
  const size_t ml_smem = (size_t)kMlWarps * 3 * S * 8;
  if (ml_smem > 48 * 1024) BPP_CUDA(cudaFuncSetAttribute(dist_ml_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ml_smem));

  // ---- 4. blocks of consecutive first leaves: counts, then ML ---------------------------------------------------------------
  const long long npairs = L * (L - 1) / 2, KK = (long long)K * K;
  const long long per_pair = KK * 4;
  const long long max_pairs = std::max<long long>(L - 1, (long long)(kCountBudget / (size_t)per_pair));
  DevMem dcnt, ddist, dlnl;
  BPP_CUDA(cudaMalloc(&dcnt.p, (size_t)std::min(npairs, max_pairs) * (size_t)per_pair));
  BPP_CUDA(cudaMalloc(&ddist.p, (size_t)npairs * 8));
  BPP_CUDA(cudaMalloc(&dlnl.p, (size_t)npairs * 8));
  const int ntiles = (int)((L * K + kTile - 1) / kTile);
  const long long nchunks = npad / kChunk;
  int occupancy = 0;
  BPP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occupancy, dist_count_kernel, 256, 0));
  const long long slots = (long long)std::max(occupancy, 1) * prop.multiProcessorCount;
  for (long long a0 = 0; a0 < L - 1;) {
    long long a1 = a0, np = 0;
    while (a1 < L - 1 && np + (L - 1 - a1) <= max_pairs) np += L - 1 - a1++;
    const long long pair_base = pair_index(a0, a0 + 1, L);
    const int ti0 = (int)(a0 * K / kTile), ti1 = (int)((a1 * K - 1) / kTile);
    long long tiles = 0;
    for (int ti = ti0; ti <= ti1; ++ti) tiles += ntiles - ti;
    const long long slices = count_slices(tiles, nchunks, slots);
    const long long per_slice = (nchunks + slices - 1) / slices;
    const dim3 grid((unsigned)ntiles, (unsigned)(ti1 - ti0 + 1), (unsigned)((nchunks + per_slice - 1) / per_slice));
    if (grid.y > 65535u || grid.z > 65535u) BPP_FAIL(BPPGPU_E_INVALID, "too many sequences x codes for the count grid");
    BPP_CUDA(cudaEventRecord(ev[0], st));
    BPP_CUDA(cudaMemsetAsync(dcnt.p, 0, (size_t)np * (size_t)per_pair, st));
    dist_count_kernel<<<grid, 256, 0, st>>>(packed.as<uint8_t>(), dw8.as<uint8_t>(), npad, (int)L, K, ti0, (int)a0, (int)a1, pair_base,
                                            per_slice, dcnt.as<unsigned>());
    BPP_CUDA(cudaGetLastError());
    BPP_CUDA(cudaEventRecord(ev[1], st));
    BPP_CUDA(elapsed(ms));
    ms_count += ms;
    MlArgs args{dcnt.as<unsigned>(), np, K, S, n_cats, dA.as<double>(), dB.as<double>(), dmu.as<double>(), drt.as<double>(),
                dpr.as<double>(), damb.as<uint8_t>(), ddist.as<double>() + pair_base, dlnl.as<double>() + pair_base};
    BPP_CUDA(cudaEventRecord(ev[0], st));
    dist_ml_kernel<<<(unsigned)((np + kMlWarps - 1) / kMlWarps), kMlWarps * 32, ml_smem, st>>>(args);
    BPP_CUDA(cudaGetLastError());
    BPP_CUDA(cudaEventRecord(ev[1], st));
    BPP_CUDA(elapsed(ms));
    ms_ml += ms;
    if (counts) BPP_CUDA(staged_copy(counts + (size_t)pair_base * KK, dcnt.p, (size_t)np * (size_t)per_pair, false, device));
    a0 = a1;
  }

  // ---- 5. symmetric matrices ------------------------------------------------------------------------------------------------
  std::vector<double> pd((size_t)npairs), pl((size_t)npairs);
  BPP_CUDA(cudaMemcpy(pd.data(), ddist.p, (size_t)npairs * 8, cudaMemcpyDeviceToHost));
  BPP_CUDA(cudaMemcpy(pl.data(), dlnl.p, (size_t)npairs * 8, cudaMemcpyDeviceToHost));
  for (long long i = 0; i < L; ++i) {
    dist[i * L + i] = 0.0;
    if (lnl) lnl[i * L + i] = 0.0;
    for (long long j = i + 1; j < L; ++j) {
      const long long p = pair_index(i, j, L);
      dist[i * L + j] = dist[j * L + i] = pd[(size_t)p];
      if (lnl) lnl[i * L + j] = lnl[j * L + i] = pl[(size_t)p];
    }
  }
  g_last_ms[0] = ms_upload;
  g_last_ms[1] = ms_count;
  g_last_ms[2] = ms_ml;
  return BPPGPU_OK;
}

int bppgpu_pairwise_distances_timing(double* upload_ms, double* count_ms, double* ml_ms) {
  if (upload_ms) *upload_ms = g_last_ms[0];
  if (count_ms) *count_ms = g_last_ms[1];
  if (ml_ms) *ml_ms = g_last_ms[2];
  return BPPGPU_OK;
}
