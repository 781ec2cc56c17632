// libbppgpu: Fitch parsimony with double-recursive arrays (Parsimony/DRTreeParsimonyScore.cpp: computeScoresFromArrays,
// testNNI).  Semantics in DESIGN.md section 7b.
//
// The handle holds the tip sets resident: one row per leaf, one element per pattern, bit x set iff code_table[code][x] > 0,
// stored as uint8 / uint16 / uint32 by the number of state bits.  The topology comes with every call (an NNI search changes it
// every round) and is flattened on the host into two programs:
//   post: the internal nodes in post-order, each with its sons in son order.  One thread owns a run of patterns and walks the
//         whole program per pattern: B = U[s_1]; B & U[s_j] == 0 ? (B |= U[s_j], c += 1) : (B &= U[s_j]).  U of every internal
//         node is written (fathers read their sons' sets back), c is the pattern's score; sum_i w_i c_i is reduced in int64.
//   pre:  the non-root internal nodes f in pre-order, with the four sides of the edge (f, g): A0, A1 = U of f's sons, C = U of
//         the uncle, X = D[g] (or U of the root's third son).  D[f] = merge(C, X) is written when a son of f reads it, and
//         both NNIs of the edge are scored from the same four sets (delta per pattern in [-3, 3], times the weight).  Here the
//         loop order is the other way round (op outer, the thread's patterns inner), so that each NNI's sum is reduced across
//         the CTA: a warp shuffle tree, then kBatch edges' warp partials in shared memory, one int64 atomic per CTA and NNI.
// Leaves' D is never read (X comes from an internal g), so only internal nodes have a D row.  Patterns are processed in
// blocks sized so that U and D of a block fit `max_bytes`; block totals add up exactly (integer sums).
#include "common.cuh"
#include "bppgpu.h"
#include "staging.h"

#include <algorithm>
#include <cstring>
#include <memory>
#include <vector>

namespace bppgpu {
namespace {

constexpr int kMaxBits = 32;
constexpr int kMaxCodes = 8192;                          // code -> set table in shared memory (32 KB)
constexpr size_t kDefaultMaxBytes = (size_t)8 << 30;     // U + D of one pattern block
constexpr int kThreads = 256;
constexpr int kBatch = 16;                               // edges whose warp partials share one __syncthreads

// a son reference: >= 0 internal slot (U row), < 0 leaf row -(r + 1) (tip set row)
template <typename T>
__device__ __forceinline__ T load_set(int ref, const T* __restrict__ tips, long long tip_stride, const T* __restrict__ U,
                                      long long nb, long long p) {
  return ref >= 0 ? U[(size_t)ref * nb + p] : tips[(size_t)(-ref - 1) * tip_stride + p];
}

template <typename T>
__device__ __forceinline__ T fitch(T a, T b, int& fail) {
  const T i = a & b;
  fail += i == 0;
  return i ? i : (T)(a | b);
}

template <typename T>
__global__ void pars_pack_kernel(const void* __restrict__ codes, int code_bytes, long long n, int n_codes,
                                 const uint32_t* __restrict__ code_sets, T* __restrict__ out, int* __restrict__ bad) {
  extern __shared__ uint32_t s_sets[];
  for (int i = threadIdx.x; i < n_codes; i += blockDim.x) s_sets[i] = code_sets[i];
  __syncthreads();
  const size_t row = (size_t)blockIdx.y * n;
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (long long)gridDim.x * blockDim.x) {
    const unsigned c = code_bytes == 1 ? static_cast<const uint8_t*>(codes)[row + j] : static_cast<const uint16_t*>(codes)[row + j];
    T s = 0;
    if (c >= (unsigned)n_codes) atomicOr(bad, 1);
    else s = (T)s_sets[c];
    out[row + j] = s;
  }
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// post-order pass over patterns [p0, p0 + nb): U of every internal node, per-pattern score, weighted total
template <typename T>
__global__ void __launch_bounds__(kThreads) pars_post_kernel(const int* __restrict__ op_off, const int* __restrict__ kids, int n_ops,
                                                            const T* __restrict__ tips, long long tip_stride,
                                                            const uint32_t* __restrict__ w, long long nb, T* __restrict__ U,
                                                            uint32_t* __restrict__ site_scores, unsigned long long* __restrict__ total) {
  __shared__ long long s_part[kThreads / 32];
  long long acc = 0;
  for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nb; p += (long long)gridDim.x * blockDim.x) {
    int fail = 0;
    for (int op = 0; op < n_ops; ++op) {
      const int k0 = __ldg(op_off + op), k1 = __ldg(op_off + op + 1);
      T b = load_set(__ldg(kids + k0), tips, tip_stride, U, nb, p);
      for (int k = k0 + 1; k < k1; ++k) b = fitch(b, load_set(__ldg(kids + k), tips, tip_stride, U, nb, p), fail);
      U[(size_t)op * nb + p] = b;
    }
    if (site_scores) site_scores[p] = (uint32_t)fail;
    acc += (long long)w[p] * fail;
  }
  acc = warp_sum_ll(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long s = 0;
    for (int i = 0; i < kThreads / 32; ++i) s += s_part[i];
    if (s) atomicAdd(total, (unsigned long long)s);
  }
}

struct PreOp {
  int f;        // U / D slot of f
  int a0, a1;   // son references of f (the two NNIs move a0, a1)
  int c;        // uncle reference
  int x;        // D slot of g, or (flags & kXIsU) the root's third son's reference
  int flags;
};
constexpr int kXIsU = 1, kWriteD = 2;

__device__ __forceinline__ int merge_fails(uint32_t p, uint32_t q, uint32_t r, uint32_t s) {
  int f = 0;
  const uint32_t a = fitch(p, q, f), b = fitch(r, s, f);
  fitch(a, b, f);
  return f;
}

// pre-order pass over patterns [0, nb) of the block: D rows and the two NNIs of every edge (f, g); nni[2 * op + j] += sum of
// w_i * (m(C, A_1-j, A_j, X) - m(A0, A1, C, X))
template <typename T>
__global__ void __launch_bounds__(kThreads) pars_pre_kernel(const PreOp* __restrict__ ops, int n_ops, const T* __restrict__ tips,
                                                           long long tip_stride, const uint32_t* __restrict__ w, long long nb,
                                                           const T* __restrict__ U, T* __restrict__ D,
                                                           unsigned long long* __restrict__ nni) {
  __shared__ long long s_part[kBatch][2][kThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (int b0 = 0; b0 < n_ops; b0 += kBatch) {
    const int b1 = min(n_ops, b0 + kBatch);
    for (int op = b0; op < b1; ++op) {
      const PreOp o = ops[op];
      long long d0 = 0, d1 = 0;
      for (long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x; p < nb; p += stride) {
        const T a0 = load_set(o.a0, tips, tip_stride, U, nb, p), a1 = load_set(o.a1, tips, tip_stride, U, nb, p);
        const T c = load_set(o.c, tips, tip_stride, U, nb, p);
        const T x = (o.flags & kXIsU) ? load_set(o.x, tips, tip_stride, U, nb, p) : D[(size_t)o.x * nb + p];
        if (o.flags & kWriteD) {
          int unused = 0;
          D[(size_t)o.f * nb + p] = fitch(c, x, unused);
        }
        const int cur = merge_fails(a0, a1, c, x);
        const long long wp = w[p];
        d0 += wp * (merge_fails(c, a1, a0, x) - cur);
        d1 += wp * (merge_fails(c, a0, a1, x) - cur);
      }
      d0 = warp_sum_ll(d0);
      d1 = warp_sum_ll(d1);
      if (lane == 0) {
        s_part[op - b0][0][warp] = d0;
        s_part[op - b0][1][warp] = d1;
      }
    }
    __syncthreads();
    if (threadIdx.x < 2 * (b1 - b0)) {
      const int e = threadIdx.x >> 1, j = threadIdx.x & 1;
      long long s = 0;
      for (int i = 0; i < kThreads / 32; ++i) s += s_part[e][j][i];
      if (s) atomicAdd(nni + 2 * (b0 + e) + j, (unsigned long long)s);
    }
    __syncthreads();
  }
}

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
  ~DevBuf() { cudaFree(p); }
  cudaError_t ensure(size_t n) {
    if (n <= bytes) return cudaSuccess;
    cudaFree(p);
    p = nullptr;
    bytes = 0;
    cudaError_t r = cudaMalloc(&p, n);
    if (r == cudaSuccess) bytes = n;
    return r;
  }
  template <typename T>
  T* as() const { return static_cast<T*>(p); }
};

// the flattened topology of one call
struct Program {
  std::vector<int> op_off, kids;      // post-order ops (internal nodes, root last)
  std::vector<PreOp> pre;             // pre-order ops (non-root internal nodes)
  std::vector<int> pre_v;             // [2 * n_pre]: node ids of a0, a1 (the NNI's v)
  int n_int = 0;
};

}  // namespace
}  // namespace bppgpu

using namespace bppgpu;

struct bppgpu_parsimony {
  int device = 0;
  int elem = 1;                 // bytes per set
  int n_leaves = 0;
  long long n_patterns = 0;
  size_t max_bytes = kDefaultMaxBytes;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  double last_ms = 0;
  DevBuf tips, weights, work, prog, scores, sums;
  ~bppgpu_parsimony() {
    if (ev[0]) cudaEventDestroy(ev[0]);
    if (ev[1]) cudaEventDestroy(ev[1]);
    if (stream) cudaStreamDestroy(stream);
  }
};

namespace {

int flatten(const bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* off, const int32_t* ch, const int32_t* leaf_row,
            bool nni, Program& pg) {
  if (n_nodes < 1 || !off || !ch || !leaf_row) BPP_FAIL(BPPGPU_E_INVALID, "bad topology arguments");
  if (root < 0 || root >= n_nodes) BPP_FAIL(BPPGPU_E_INVALID, "root %d out of range (0..%d)", root, n_nodes - 1);
  if (off[0] != 0) BPP_FAIL(BPPGPU_E_INVALID, "child_offsets[0] must be 0");
  for (int i = 0; i < n_nodes; ++i)
    if (off[i + 1] < off[i]) BPP_FAIL(BPPGPU_E_INVALID, "child_offsets must not decrease (node %d)", i);
  if (off[root + 1] == off[root]) BPP_FAIL(BPPGPU_E_INVALID, "the root must have sons");
  // every node reached exactly once from the root; post-order by an explicit stack
  std::vector<int> father(n_nodes, -2), post;
  post.reserve(n_nodes);
  father[root] = -1;
  std::vector<std::pair<int, int> > st{{root, 0}};
  while (!st.empty()) {
    const int v = st.back().first, k = off[v] + st.back().second;
    if (k < off[v + 1]) {
      ++st.back().second;
      const int s = ch[k];
      if (s < 0 || s >= n_nodes) BPP_FAIL(BPPGPU_E_INVALID, "son %d of node %d out of range", s, v);
      if (father[s] != -2) BPP_FAIL(BPPGPU_E_INVALID, "node %d is reached twice from the root", s);
      father[s] = v;
      st.push_back({s, 0});
    } else {
      post.push_back(v);
      st.pop_back();
    }
  }
  if ((int)post.size() != n_nodes) BPP_FAIL(BPPGPU_E_INVALID, "%d of %d nodes are not reached from the root", n_nodes - (int)post.size(), n_nodes);
  std::vector<char> used(h->n_leaves, 0);
  std::vector<int> slot(n_nodes, -1);
  for (int v : post) {
    if (off[v + 1] > off[v]) { slot[v] = pg.n_int++; continue; }
    const int r = leaf_row[v];
    if (r < 0 || r >= h->n_leaves) BPP_FAIL(BPPGPU_E_INVALID, "leaf %d has tip row %d (0..%d)", v, r, h->n_leaves - 1);
    if (used[r]) BPP_FAIL(BPPGPU_E_INVALID, "tip row %d is named by two leaves", r);
    used[r] = 1;
  }
  auto ref = [&](int v) { return slot[v] >= 0 ? slot[v] : -(leaf_row[v] + 1); };
  pg.op_off.assign(1, 0);
  for (int v : post) {
    if (slot[v] < 0) continue;
    for (int k = off[v]; k < off[v + 1]; ++k) pg.kids.push_back(ref(ch[k]));
    pg.op_off.push_back((int)pg.kids.size());
  }
  if (!nni) return BPPGPU_OK;
  for (int v : post) {
    const int ns = off[v + 1] - off[v];
    if (v == root ? ns != 3 : (ns != 0 && ns != 2))
      BPP_FAIL(BPPGPU_E_INVALID, "NNI scoring needs a binary topology with a three-son root (node %d has %d sons)", v, ns);
  }
  // pre-order = reversed post-order with sons in reverse: any order with fathers before sons will do
  for (auto it = post.rbegin(); it != post.rend(); ++it) {
    const int f = *it;
    if (f == root || slot[f] < 0) continue;
    const int g = father[f];
    const int ng = off[g + 1] - off[g];
    int pos = 0;
    while (ch[off[g] + pos] != f) ++pos;
    const int u = ch[off[g] + (pos > 1 ? 0 : 1 - pos)];
    PreOp o;
    o.f = slot[f];
    o.a0 = ref(ch[off[f]]);
    o.a1 = ref(ch[off[f] + 1]);
    o.c = ref(u);
    o.flags = 0;
    if (g == root) {
      int third = -1;
      for (int k = 0; k < ng; ++k)
        if (ch[off[g] + k] != f && ch[off[g] + k] != u) third = ch[off[g] + k];
      o.x = ref(third);
      o.flags |= kXIsU;
    } else {
      o.x = slot[g];
    }
    if (slot[ch[off[f]]] >= 0 || slot[ch[off[f] + 1]] >= 0) o.flags |= kWriteD;
    pg.pre.push_back(o);
    pg.pre_v.push_back(ch[off[f]]);
    pg.pre_v.push_back(ch[off[f] + 1]);
  }
  return BPPGPU_OK;
}

template <typename T>
int run_passes(bppgpu_parsimony* h, const Program& pg, bool nni, long long nb_max, uint32_t* site_scores_dev) {
  cudaStream_t st = h->stream;
  const int n_post = (int)pg.op_off.size() - 1, n_pre = (int)pg.pre.size();
  const int* d_off = h->prog.as<int>();
  const int* d_kids = d_off + pg.op_off.size();
  const PreOp* d_pre = reinterpret_cast<const PreOp*>(h->prog.as<char>() + (((pg.op_off.size() + pg.kids.size()) * 4 + 15) / 16 * 16));
  T* U = h->work.as<T>();
  T* D = U + (size_t)pg.n_int * nb_max;
  unsigned long long* total = h->sums.as<unsigned long long>();
  int sms = 0, occ = 0;
  BPP_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, h->device));
  BPP_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pars_pre_kernel<T>, kThreads, 0));
  for (long long p0 = 0; p0 < h->n_patterns; p0 += nb_max) {
    const long long nb = std::min(nb_max, h->n_patterns - p0);
    const T* tips = h->tips.as<T>() + p0;
    const uint32_t* w = h->weights.as<uint32_t>() + p0;
    const long long blocks = (nb + kThreads - 1) / kThreads;
    pars_post_kernel<T><<<(unsigned)std::min<long long>(blocks, 1 << 20), kThreads, 0, st>>>(
        d_off, d_kids, n_post, tips, h->n_patterns, w, nb, U, site_scores_dev ? site_scores_dev + p0 : nullptr, total);
    BPP_CUDA(cudaGetLastError());
    if (nni && n_pre > 0) {
      // one wave: each thread keeps its patterns for the whole program, so the per-edge CTA reductions are as few as possible
      const long long grid = std::min<long long>(blocks, (long long)std::max(occ, 1) * sms);
      pars_pre_kernel<T><<<(unsigned)grid, kThreads, 0, st>>>(d_pre, n_pre, tips, h->n_patterns, w, nb, U, D, total + 1);
      BPP_CUDA(cudaGetLastError());
    }
  }
  return BPPGPU_OK;
}

int run(bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* off, const int32_t* ch, const int32_t* leaf_row,
        bool nni, int64_t* delta, int64_t* score, uint32_t* site_scores) {
  if (!h) BPP_FAIL(BPPGPU_E_INVALID, "null parsimony handle");
  Program pg;
  int rc = flatten(h, n_nodes, root, off, ch, leaf_row, nni, pg);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  // U and D rows per pattern; the block is the most patterns whose rows fit max_bytes
  const size_t per_pattern = (size_t)pg.n_int * (nni ? 2 : 1) * h->elem;
  const long long nb_max = std::max<long long>(1, std::min<long long>(h->n_patterns, (long long)(h->max_bytes / per_pattern)));
  BPP_CUDA(h->work.ensure(per_pattern * (size_t)nb_max));
  const size_t pre_at = ((pg.op_off.size() + pg.kids.size()) * 4 + 15) / 16 * 16;
  std::vector<char> img(pre_at + pg.pre.size() * sizeof(PreOp));
  std::memcpy(img.data(), pg.op_off.data(), pg.op_off.size() * 4);
  std::memcpy(img.data() + pg.op_off.size() * 4, pg.kids.data(), pg.kids.size() * 4);
  if (!pg.pre.empty()) std::memcpy(img.data() + pre_at, pg.pre.data(), pg.pre.size() * sizeof(PreOp));
  BPP_CUDA(h->prog.ensure(img.size()));
  const size_t n_sums = 1 + pg.pre.size() * 2;
  BPP_CUDA(h->sums.ensure(n_sums * 8));
  if (site_scores) BPP_CUDA(h->scores.ensure((size_t)h->n_patterns * 4));
  BPP_CUDA(cudaMemcpyAsync(h->prog.p, img.data(), img.size(), cudaMemcpyHostToDevice, st));
  BPP_CUDA(cudaMemsetAsync(h->sums.p, 0, n_sums * 8, st));
  BPP_CUDA(cudaEventRecord(h->ev[0], st));
  uint32_t* dsc = site_scores ? h->scores.as<uint32_t>() : nullptr;
  if (h->elem == 1) rc = run_passes<uint8_t>(h, pg, nni, nb_max, dsc);
  else if (h->elem == 2) rc = run_passes<uint16_t>(h, pg, nni, nb_max, dsc);
  else rc = run_passes<uint32_t>(h, pg, nni, nb_max, dsc);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(cudaEventRecord(h->ev[1], st));
  std::vector<long long> sums(n_sums);
  BPP_CUDA(cudaMemcpyAsync(sums.data(), h->sums.p, n_sums * 8, cudaMemcpyDeviceToHost, st));
  BPP_CUDA(cudaStreamSynchronize(st));
  float ms = 0;
  BPP_CUDA(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
  h->last_ms = ms;
  if (site_scores) BPP_CUDA(staged_copy(site_scores, h->scores.p, (size_t)h->n_patterns * 4, false, h->device));
  if (score) *score = sums[0];
  if (delta) {
    std::fill(delta, delta + n_nodes, (int64_t)0);
    for (size_t i = 0; i < pg.pre_v.size(); ++i) delta[pg.pre_v[i]] = sums[1 + i];
  }
  return BPPGPU_OK;
}

}  // namespace

int bppgpu_parsimony_create(int device, int32_t n_states, int32_t n_codes, int32_t code_bytes, const double* code_table,
                            int32_t n_leaves, int64_t n_patterns, const void* tip_codes, const uint32_t* weights, int64_t max_bytes,
                            bppgpu_parsimony** out) {
  if (!out || !code_table || !tip_codes || !weights || n_patterns < 1 || max_bytes < 0)
    BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_parsimony_create");
  *out = nullptr;
  if (n_states < 1 || n_states > kMaxBits)
    BPP_FAIL(BPPGPU_E_INVALID, "parsimony sets hold 1..%d states, got %d (codon and chromosome alphabets are too large)", kMaxBits, n_states);
  if (n_codes < 1 || n_codes > kMaxCodes) BPP_FAIL(BPPGPU_E_INVALID, "parsimony takes 1..%d tip codes, got %d", kMaxCodes, n_codes);
  if (code_bytes != 1 && code_bytes != 2) BPP_FAIL(BPPGPU_E_INVALID, "code_bytes must be 1 or 2");
  if (n_leaves < 2 || n_leaves > 65535) BPP_FAIL(BPPGPU_E_INVALID, "parsimony needs 2..65535 sequences, got %d", n_leaves);
  std::vector<uint32_t> sets(n_codes, 0);
  for (int c = 0; c < n_codes; ++c) {
    for (int x = 0; x < n_states; ++x)
      if (code_table[(size_t)c * n_states + x] > 0) sets[c] |= 1u << x;
    if (!sets[c]) BPP_FAIL(BPPGPU_E_INVALID, "code %d has no positive entry in the code table (an empty Fitch set)", c);
  }
  int ndev = 0;
  cudaError_t r = cudaGetDeviceCount(&ndev);
  if (r != cudaSuccess || ndev == 0)
    BPP_FAIL(BPPGPU_E_CUDA, "no usable CUDA device (%s); libbppgpu has no CPU fallback", r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
  if (device < 0 || device >= ndev) BPP_FAIL(BPPGPU_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  BPP_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BPP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) BPP_FAIL(BPPGPU_E_CUDA, "device %d is sm_%d%d; libbppgpu is built for sm_100a only", device, prop.major, prop.minor);

  std::unique_ptr<bppgpu_parsimony> h(new bppgpu_parsimony());
  h->device = device;
  h->elem = n_states <= 8 ? 1 : n_states <= 16 ? 2 : 4;
  h->n_leaves = n_leaves;
  h->n_patterns = n_patterns;
  if (max_bytes > 0) h->max_bytes = (size_t)max_bytes;
  BPP_CUDA(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
  BPP_CUDA(cudaEventCreate(&h->ev[0]));
  BPP_CUDA(cudaEventCreate(&h->ev[1]));
  cudaStream_t st = h->stream;
  const size_t L = (size_t)n_leaves, N = (size_t)n_patterns;
  BPP_CUDA(h->weights.ensure(N * 4));
  BPP_CUDA(cudaMemcpy(h->weights.p, weights, N * 4, cudaMemcpyDefault));
  // tip codes on the device (read in place when they already are), packed to set rows
  cudaPointerAttributes at;
  const bool resident = cudaPointerGetAttributes(&at, tip_codes) == cudaSuccess && at.type == cudaMemoryTypeDevice && at.device == device;
  cudaGetLastError();
  DevBuf raw, dsets, dbad;
  const void* src = tip_codes;
  if (!resident) {
    BPP_CUDA(raw.ensure(L * N * code_bytes));
    BPP_CUDA(staged_copy(raw.p, tip_codes, L * N * code_bytes, true, device));
    src = raw.p;
  }
  BPP_CUDA(h->tips.ensure(L * N * h->elem));
  BPP_CUDA(dsets.ensure((size_t)n_codes * 4));
  BPP_CUDA(dbad.ensure(4));
  BPP_CUDA(cudaMemcpyAsync(dsets.p, sets.data(), (size_t)n_codes * 4, cudaMemcpyHostToDevice, st));
  BPP_CUDA(cudaMemsetAsync(dbad.p, 0, 4, st));
  const dim3 grid((unsigned)std::min<size_t>((N + 255) / 256, 4096), (unsigned)L);
  const size_t smem = (size_t)n_codes * 4;
  if (h->elem == 1)
    pars_pack_kernel<uint8_t><<<grid, 256, smem, st>>>(src, code_bytes, n_patterns, n_codes, dsets.as<uint32_t>(), h->tips.as<uint8_t>(), dbad.as<int>());
  else if (h->elem == 2)
    pars_pack_kernel<uint16_t><<<grid, 256, smem, st>>>(src, code_bytes, n_patterns, n_codes, dsets.as<uint32_t>(), h->tips.as<uint16_t>(), dbad.as<int>());
  else
    pars_pack_kernel<uint32_t><<<grid, 256, smem, st>>>(src, code_bytes, n_patterns, n_codes, dsets.as<uint32_t>(), h->tips.as<uint32_t>(), dbad.as<int>());
  BPP_CUDA(cudaGetLastError());
  int bad = 0;
  BPP_CUDA(cudaMemcpyAsync(&bad, dbad.p, 4, cudaMemcpyDeviceToHost, st));
  BPP_CUDA(cudaStreamSynchronize(st));
  if (bad) BPP_FAIL(BPPGPU_E_INVALID, "a tip code is >= n_codes (%d)", n_codes);
  *out = h.release();
  return BPPGPU_OK;
}

int bppgpu_parsimony_score(bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* children,
                           const int32_t* leaf_row, int64_t* score, uint32_t* site_scores) {
  if (!score) BPP_FAIL(BPPGPU_E_INVALID, "score must not be NULL");
  return run(h, n_nodes, root, child_offsets, children, leaf_row, false, nullptr, score, site_scores);
}

int bppgpu_parsimony_nni(bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* children,
                         const int32_t* leaf_row, int64_t* delta, int64_t* score) {
  if (!delta) BPP_FAIL(BPPGPU_E_INVALID, "delta must not be NULL");
  return run(h, n_nodes, root, child_offsets, children, leaf_row, true, delta, score, nullptr);
}

int bppgpu_parsimony_last_ms(bppgpu_parsimony* h, double* ms) {
  if (!h || !ms) BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_parsimony_last_ms");
  *ms = h->last_ms;
  return BPPGPU_OK;
}

int bppgpu_parsimony_destroy(bppgpu_parsimony* h) {
  if (h) {
    cudaSetDevice(h->device);
    delete h;
  }
  return BPPGPU_OK;
}
