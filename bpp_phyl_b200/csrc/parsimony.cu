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
//
// A call scores a batch of entries: entry e is one topology under one weight row (a bootstrap replicate's, or the handle's own
// for bppgpu_parsimony_score / _nni, which are the batch of one).  The entries' programs are concatenated, with U / D slots
// numbered across the batch, so the passes index U and D as for one topology.  A CTA serves one entry: blockIdx.x = entry,
// blockIdx.y = pattern chunk, so that the entries of a chunk are next to each other in launch order.  The intent is that a
// chunk of tip sets comes from HBM about once and from L2 for the other entries; no DRAM or L2 counter has been read.  At
// 1024 taxa x 1M patterns the batched calls' device time per entry is no lower than a single call's (DESIGN 7b), so no such
// reuse shows in time there (the uint8 passes are instruction-bound).  The entry comes from blockIdx.x rather than a
// division of a 1D index: with the division, nvcc gave the pre pass 32 registers instead of 64, and both passes ran slower.
//
// Bootstrap replicate weights (bppgpu_bootstrap_weights): draw j of replicate R is Philox4x32-10 (Salmon et al. 2011, as in
// Random123) with key (seed lo, seed hi) and counter (j lo, j hi, R, 0); u = x0 | x1 << 32 draws site floor(u * n_sites / 2^64).
#include "common.cuh"
#include "bppgpu.h"
#include "philox.cuh"
#include "staging.h"

#include <algorithm>
#include <cstring>
#include <memory>
#include <string>
#include <vector>

namespace bppgpu {
namespace {

constexpr int kMaxBits = 32;
constexpr int kMaxCodes = 8192;                          // code -> set table in shared memory (32 KB)
constexpr size_t kDefaultMaxBytes = (size_t)8 << 30;     // U + D of one pattern block
constexpr int kThreads = 256;
constexpr int kBatch = 16;                               // edges whose warp partials share one __syncthreads
constexpr long long kMaxChunks = 65535;                  // pattern chunks per launch (gridDim.y); more loop in the kernel

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

// one entry of a batch: its ops in the concatenated programs, its weight row, and its sums (score at sums[entry], the NNI
// sums of its pre-order op i at sums[n_entries + 2 * (pre_op + i) + j])
struct Entry {
  int post_op, n_post;   // post-order ops [post_op, post_op + n_post) (their U slots are the same numbers)
  int pre_op, n_pre;     // pre-order ops [pre_op, pre_op + n_pre)
  long long w_row;       // offset of the entry's weight row
};

// post-order pass over patterns [p0, p0 + nb): U of every internal node, per-pattern score, weighted total; one entry per CTA.
// Full occupancy (32 registers): without the bound nvcc takes 40 for 16-bit sets.
template <typename T>
__global__ void __launch_bounds__(kThreads, 2048 / kThreads) pars_post_kernel(const Entry* __restrict__ ent, const int* __restrict__ op_off,
                                                            const int* __restrict__ kids, const T* __restrict__ tips,
                                                            long long tip_stride, const uint32_t* __restrict__ w, long long nb,
                                                            T* __restrict__ U, uint32_t* __restrict__ site_scores,
                                                            long long score_stride, unsigned long long* __restrict__ total) {
  __shared__ long long s_part[kThreads / 32];
  const int e = blockIdx.x;
  const Entry en = ent[e];
  const uint32_t* we = w + en.w_row;
  long long acc = 0;
  for (long long p = (long long)blockIdx.y * blockDim.x + threadIdx.x; p < nb; p += (long long)gridDim.y * blockDim.x) {
    int fail = 0;
    for (int op = en.post_op; op < en.post_op + en.n_post; ++op) {
      const int k0 = __ldg(op_off + op), k1 = __ldg(op_off + op + 1);
      T b = load_set(__ldg(kids + k0), tips, tip_stride, U, nb, p);
      for (int k = k0 + 1; k < k1; ++k) b = fitch(b, load_set(__ldg(kids + k), tips, tip_stride, U, nb, p), fail);
      U[(size_t)op * nb + p] = b;
    }
    if (site_scores) site_scores[(size_t)e * score_stride + p] = (uint32_t)fail;
    acc += (long long)we[p] * fail;
  }
  acc = warp_sum_ll(acc);
  if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    long long s = 0;
    for (int i = 0; i < kThreads / 32; ++i) s += s_part[i];
    if (s) atomicAdd(total + e, (unsigned long long)s);
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
// w_i * (m(C, A_1-j, A_j, X) - m(A0, A1, C, X)); one entry per CTA
template <typename T>
__global__ void __launch_bounds__(kThreads) pars_pre_kernel(const Entry* __restrict__ ent, const PreOp* __restrict__ ops,
                                                           const T* __restrict__ tips, long long tip_stride,
                                                           const uint32_t* __restrict__ w, long long nb, const T* __restrict__ U,
                                                           T* __restrict__ D, unsigned long long* __restrict__ nni) {
  __shared__ long long s_part[kBatch][2][kThreads / 32];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const Entry en = ent[blockIdx.x];
  const long long stride = (long long)gridDim.y * blockDim.x;
  const long long p_first = (long long)blockIdx.y * blockDim.x + threadIdx.x;
  const uint32_t* we = w + en.w_row;
  const int n_ops = en.n_pre;
  ops += en.pre_op;           // the entry's ops and sums, indexed from 0
  nni += 2 * (size_t)en.pre_op;
  for (int b0 = 0; b0 < n_ops; b0 += kBatch) {
    const int b1 = min(n_ops, b0 + kBatch);
    for (int op = b0; op < b1; ++op) {
      const PreOp o = ops[op];
      long long d0 = 0, d1 = 0;
      for (long long p = p_first; p < nb; p += stride) {
        const T a0 = load_set(o.a0, tips, tip_stride, U, nb, p), a1 = load_set(o.a1, tips, tip_stride, U, nb, p);
        const T c = load_set(o.c, tips, tip_stride, U, nb, p);
        const T x = (o.flags & kXIsU) ? load_set(o.x, tips, tip_stride, U, nb, p) : D[(size_t)o.x * nb + p];
        if (o.flags & kWriteD) {
          int unused = 0;
          D[(size_t)o.f * nb + p] = fitch(c, x, unused);
        }
        const int cur = merge_fails(a0, a1, c, x);
        const long long wp = we[p];
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

// ---- bootstrap replicate weights ----------------------------------------------------------------------------------------------
__global__ void boot_check_kernel(const int64_t* __restrict__ idx, long long n_sites, long long n_patterns, int* __restrict__ bad) {
  for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < n_sites; j += (long long)gridDim.x * blockDim.x)
    if (idx[j] < 0 || idx[j] >= n_patterns) atomicOr(bad, 1);
}

// w[r][idx[site]] += 1 for every draw (j, r) of replicates first .. first + n_reps - 1
__global__ void boot_draw_kernel(const int64_t* __restrict__ idx, unsigned long long n_sites, long long n_patterns, uint32_t first,
                                 unsigned long long n_draws, uint64_t seed, uint32_t* __restrict__ w) {
  for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_draws;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    const unsigned long long r = i / n_sites, j = i - r * n_sites;
    uint32_t c[4] = {(uint32_t)j, (uint32_t)(j >> 32), first + (uint32_t)r, 0u};
    philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
    const unsigned long long u = (unsigned long long)c[0] | (unsigned long long)c[1] << 32;
    atomicAdd(w + r * n_patterns + idx[__umul64hi(u, n_sites)], 1u);
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
  int n_reps = 0;               // replicate weight rows in `reps`
  DevBuf tips, weights, reps, work, prog, scores, sums;
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
  // a tree has n_nodes - 1 sons in all; this also keeps the reads of `children` inside an entry's row of a batch
  if (off[n_nodes] != n_nodes - 1) BPP_FAIL(BPPGPU_E_INVALID, "child_offsets[n_nodes] is %d, a tree has %d sons", off[n_nodes], n_nodes - 1);
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

// appends one entry's program to the batch's, numbering its U / D slots after those already there
void append(Program& all, const Program& one) {
  const int base = all.n_int;
  auto rebase = [base](int ref) { return ref >= 0 ? ref + base : ref; };
  for (size_t i = 0; i + 1 < one.op_off.size(); ++i) {
    for (int k = one.op_off[i]; k < one.op_off[i + 1]; ++k) all.kids.push_back(rebase(one.kids[k]));
    all.op_off.push_back((int)all.kids.size());
  }
  for (PreOp o : one.pre) {
    o.f += base;
    o.a0 = rebase(o.a0);
    o.a1 = rebase(o.a1);
    o.c = rebase(o.c);
    o.x = (o.flags & kXIsU) ? rebase(o.x) : o.x + base;
    all.pre.push_back(o);
  }
  all.pre_v.insert(all.pre_v.end(), one.pre_v.begin(), one.pre_v.end());
  all.n_int += one.n_int;
}

// a batch of topologies sharing n_nodes and root: entry e reads child_offsets [e][n_nodes + 1], children [e][n_nodes - 1],
// leaf_row [e][n_nodes] and weight row rep[e] of `w` ([n_rows][n_patterns], device)
struct Batch {
  int n = 1;
  int32_t n_nodes = 0, root = 0;
  const int32_t *off = nullptr, *ch = nullptr, *leaf_row = nullptr, *rep = nullptr;
  const uint32_t* w = nullptr;
  int n_rows = 1;
  bool name_entries = false;    // error messages name the bad entry
};

template <typename T>
int run_passes(bppgpu_parsimony* h, const Program& pg, const Entry* d_ent, int n_ent, const uint32_t* w, bool nni, long long nb_max,
               uint32_t* site_scores_dev) {
  cudaStream_t st = h->stream;
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
    const long long blocks = (nb + kThreads - 1) / kThreads;
    // blockIdx.x = entry, blockIdx.y = pattern chunk: the entries of a chunk are adjacent in launch order
    const dim3 grid((unsigned)n_ent, (unsigned)std::min<long long>(blocks, kMaxChunks));
    pars_post_kernel<T><<<grid, kThreads, 0, st>>>(d_ent, d_off, d_kids, tips, h->n_patterns, w + p0, nb, U,
                                                                          site_scores_dev ? site_scores_dev + p0 : nullptr,
                                                                          h->n_patterns, total);
    BPP_CUDA(cudaGetLastError());
    if (nni && !pg.pre.empty()) {
      // one wave, split across the entries: each thread keeps its patterns for the whole program, so the per-edge CTA
      // reductions are as few as possible
      const long long pre_chunks = std::max<long long>(
          1, std::min<long long>(std::min<long long>(blocks, kMaxChunks), (long long)std::max(occ, 1) * sms / n_ent));
      pars_pre_kernel<T><<<dim3((unsigned)n_ent, (unsigned)pre_chunks), kThreads, 0, st>>>(d_ent, d_pre, tips, h->n_patterns, w + p0, nb, U, D,
                                                                               total + n_ent);
      BPP_CUDA(cudaGetLastError());
    }
  }
  return BPPGPU_OK;
}

int run(bppgpu_parsimony* h, const Batch& b, bool nni, int64_t* delta, int64_t* score, uint32_t* site_scores) {
  if (!h) BPP_FAIL(BPPGPU_E_INVALID, "null parsimony handle");
  if (b.n < 1) BPP_FAIL(BPPGPU_E_INVALID, "a batch needs at least one entry, got %d", b.n);
  if (b.n_nodes < 1 || !b.off || !b.ch || !b.leaf_row) BPP_FAIL(BPPGPU_E_INVALID, "bad topology arguments");
  Program pg;
  pg.op_off.assign(1, 0);
  std::vector<Entry> ents(b.n);
  for (int e = 0; e < b.n; ++e) {
    const int r = b.rep ? b.rep[e] : 0;
    if (r < 0 || r >= b.n_rows) BPP_FAIL(BPPGPU_E_INVALID, "entry %d: replicate %d out of range (0..%d)", e, r, b.n_rows - 1);
    Program one;
    const size_t n = (size_t)b.n_nodes;
    int rc = flatten(h, b.n_nodes, b.root, b.off + e * (n + 1), b.ch + e * (n - 1), b.leaf_row + e * n, nni, one);
    if (rc != BPPGPU_OK) {
      if (b.name_entries) last_error() = "entry " + std::to_string(e) + ": " + last_error();
      return rc;
    }
    ents[e] = Entry{(int)pg.op_off.size() - 1, one.n_int, (int)pg.pre.size(), (int)one.pre.size(), (long long)r * h->n_patterns};
    append(pg, one);
  }
  BPP_CUDA(cudaSetDevice(h->device));
  cudaStream_t st = h->stream;
  // U and D rows per pattern over all entries; the block is the most patterns whose rows fit max_bytes
  const size_t per_pattern = (size_t)pg.n_int * (nni ? 2 : 1) * h->elem;
  const long long nb_max = std::max<long long>(1, std::min<long long>(h->n_patterns, (long long)(h->max_bytes / per_pattern)));
  BPP_CUDA(h->work.ensure(per_pattern * (size_t)nb_max));
  const size_t pre_at = ((pg.op_off.size() + pg.kids.size()) * 4 + 15) / 16 * 16;
  const size_t ent_at = (pre_at + pg.pre.size() * sizeof(PreOp) + 15) / 16 * 16;
  std::vector<char> img(ent_at + ents.size() * sizeof(Entry));
  std::memcpy(img.data(), pg.op_off.data(), pg.op_off.size() * 4);
  std::memcpy(img.data() + pg.op_off.size() * 4, pg.kids.data(), pg.kids.size() * 4);
  if (!pg.pre.empty()) std::memcpy(img.data() + pre_at, pg.pre.data(), pg.pre.size() * sizeof(PreOp));
  std::memcpy(img.data() + ent_at, ents.data(), ents.size() * sizeof(Entry));
  BPP_CUDA(h->prog.ensure(img.size()));
  const Entry* d_ent = reinterpret_cast<const Entry*>(h->prog.as<char>() + ent_at);
  const size_t n_sums = b.n + pg.pre.size() * 2;
  BPP_CUDA(h->sums.ensure(n_sums * 8));
  const size_t score_bytes = (size_t)b.n * h->n_patterns * 4;
  if (site_scores) BPP_CUDA(h->scores.ensure(score_bytes));
  BPP_CUDA(cudaMemcpyAsync(h->prog.p, img.data(), img.size(), cudaMemcpyHostToDevice, st));
  BPP_CUDA(cudaMemsetAsync(h->sums.p, 0, n_sums * 8, st));
  BPP_CUDA(cudaEventRecord(h->ev[0], st));
  uint32_t* dsc = site_scores ? h->scores.as<uint32_t>() : nullptr;
  int rc;
  if (h->elem == 1) rc = run_passes<uint8_t>(h, pg, d_ent, b.n, b.w, nni, nb_max, dsc);
  else if (h->elem == 2) rc = run_passes<uint16_t>(h, pg, d_ent, b.n, b.w, nni, nb_max, dsc);
  else rc = run_passes<uint32_t>(h, pg, d_ent, b.n, b.w, nni, nb_max, dsc);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(cudaEventRecord(h->ev[1], st));
  std::vector<long long> sums(n_sums);
  BPP_CUDA(cudaMemcpyAsync(sums.data(), h->sums.p, n_sums * 8, cudaMemcpyDeviceToHost, st));
  BPP_CUDA(cudaStreamSynchronize(st));
  float ms = 0;
  BPP_CUDA(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
  h->last_ms = ms;
  if (site_scores) BPP_CUDA(staged_copy(site_scores, h->scores.p, score_bytes, false, h->device));
  if (score) std::copy(sums.begin(), sums.begin() + b.n, score);
  if (delta) {
    std::fill(delta, delta + (size_t)b.n * b.n_nodes, (int64_t)0);
    for (int e = 0; e < b.n; ++e)
      for (int i = 2 * ents[e].pre_op; i < 2 * (ents[e].pre_op + ents[e].n_pre); ++i)
        delta[(size_t)e * b.n_nodes + pg.pre_v[i]] = sums[b.n + i];
  }
  return BPPGPU_OK;
}

int check_device(int device) {
  int ndev = 0;
  cudaError_t r = cudaGetDeviceCount(&ndev);
  if (r != cudaSuccess || ndev == 0)
    BPP_FAIL(BPPGPU_E_CUDA, "no usable CUDA device (%s); libbppgpu has no CPU fallback", r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
  if (device < 0 || device >= ndev) BPP_FAIL(BPPGPU_E_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
  return BPPGPU_OK;
}

// replicate weights [n_reps][n_patterns] into device memory `out` on `st`; indices from host, pinned or device memory
int draw_weights(int device, cudaStream_t st, int64_t n_sites, const int64_t* indices, int64_t n_patterns, int64_t first,
                 int64_t n_reps, uint64_t seed, uint32_t* out, cudaEvent_t t0, cudaEvent_t t1) {
  if (!indices || n_patterns < 1) BPP_FAIL(BPPGPU_E_INVALID, "bad argument to the bootstrap sampler");
  if (n_sites < 1 || n_sites >= ((int64_t)1 << 32)) BPP_FAIL(BPPGPU_E_INVALID, "n_sites must be in 1 .. 2^32 - 1, got %lld", (long long)n_sites);
  if (n_reps < 1 || first < 0 || first + n_reps > ((int64_t)1 << 32))
    BPP_FAIL(BPPGPU_E_INVALID, "replicates %lld .. %lld: need n_replicates >= 1 and indices in 0 .. 2^32 - 1", (long long)first,
             (long long)(first + n_reps - 1));
  DevBuf didx, dbad;
  BPP_CUDA(didx.ensure((size_t)n_sites * 8));
  BPP_CUDA(dbad.ensure(4));
  BPP_CUDA(staged_copy(didx.p, indices, (size_t)n_sites * 8, true, device));
  BPP_CUDA(cudaMemsetAsync(dbad.p, 0, 4, st));
  BPP_CUDA(cudaMemsetAsync(out, 0, (size_t)n_reps * n_patterns * 4, st));
  if (t0) BPP_CUDA(cudaEventRecord(t0, st));
  boot_check_kernel<<<(unsigned)std::min<int64_t>((n_sites + 255) / 256, 4096), 256, 0, st>>>(didx.as<int64_t>(), n_sites, n_patterns,
                                                                                              dbad.as<int>());
  BPP_CUDA(cudaGetLastError());
  int bad = 0;
  BPP_CUDA(cudaMemcpyAsync(&bad, dbad.p, 4, cudaMemcpyDeviceToHost, st));
  BPP_CUDA(cudaStreamSynchronize(st));
  if (bad) BPP_FAIL(BPPGPU_E_INVALID, "a site index is outside 0 .. n_patterns - 1 (%lld)", (long long)n_patterns - 1);
  const unsigned long long n_draws = (unsigned long long)n_sites * (unsigned long long)n_reps;
  boot_draw_kernel<<<(unsigned)std::min<unsigned long long>((n_draws + 255) / 256, 1 << 16), 256, 0, st>>>(
      didx.as<int64_t>(), (unsigned long long)n_sites, n_patterns, (uint32_t)first, n_draws, seed, out);
  BPP_CUDA(cudaGetLastError());
  if (t1) BPP_CUDA(cudaEventRecord(t1, st));
  BPP_CUDA(cudaStreamSynchronize(st));
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

namespace {

// the handle's own weights: the batch of one
Batch one_topology(const bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* off, const int32_t* ch, const int32_t* leaf_row) {
  Batch b;
  b.n_nodes = n_nodes;
  b.root = root;
  b.off = off;
  b.ch = ch;
  b.leaf_row = leaf_row;
  b.w = h ? h->weights.as<uint32_t>() : nullptr;
  return b;
}

Batch replicate_batch(const bppgpu_parsimony* h, int32_t n_entries, const int32_t* rep, int32_t n_nodes, int32_t root, const int32_t* off,
                      const int32_t* ch, const int32_t* leaf_row) {
  Batch b = one_topology(h, n_nodes, root, off, ch, leaf_row);
  b.n = n_entries;
  b.rep = rep;
  b.w = h ? h->reps.as<uint32_t>() : nullptr;
  b.n_rows = h ? h->n_reps : 0;
  b.name_entries = true;
  return b;
}

}  // namespace

int bppgpu_parsimony_score(bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* children,
                           const int32_t* leaf_row, int64_t* score, uint32_t* site_scores) {
  if (!score) BPP_FAIL(BPPGPU_E_INVALID, "score must not be NULL");
  return run(h, one_topology(h, n_nodes, root, child_offsets, children, leaf_row), false, nullptr, score, site_scores);
}

int bppgpu_parsimony_nni(bppgpu_parsimony* h, int32_t n_nodes, int32_t root, const int32_t* child_offsets, const int32_t* children,
                         const int32_t* leaf_row, int64_t* delta, int64_t* score) {
  if (!delta) BPP_FAIL(BPPGPU_E_INVALID, "delta must not be NULL");
  return run(h, one_topology(h, n_nodes, root, child_offsets, children, leaf_row), true, delta, score, nullptr);
}

int bppgpu_parsimony_set_replicate_weights(bppgpu_parsimony* h, int32_t n_replicates, const uint32_t* weights) {
  if (!h || n_replicates < 0 || (n_replicates > 0 && !weights)) BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_parsimony_set_replicate_weights");
  BPP_CUDA(cudaSetDevice(h->device));
  h->n_reps = 0;
  if (n_replicates == 0) {
    cudaFree(h->reps.p);
    h->reps.p = nullptr;
    h->reps.bytes = 0;
    return BPPGPU_OK;
  }
  const size_t bytes = (size_t)n_replicates * h->n_patterns * 4;
  BPP_CUDA(h->reps.ensure(bytes));
  BPP_CUDA(staged_copy(h->reps.p, weights, bytes, true, h->device));
  h->n_reps = n_replicates;
  return BPPGPU_OK;
}

int bppgpu_parsimony_draw_replicate_weights(bppgpu_parsimony* h, int64_t n_sites, const int64_t* indices, int64_t first_replicate,
                                            int32_t n_replicates, uint64_t seed) {
  if (!h || n_replicates < 1) BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_parsimony_draw_replicate_weights");
  BPP_CUDA(cudaSetDevice(h->device));
  h->n_reps = 0;
  BPP_CUDA(h->reps.ensure((size_t)n_replicates * h->n_patterns * 4));
  int rc = draw_weights(h->device, h->stream, n_sites, indices, h->n_patterns, first_replicate, n_replicates, seed, h->reps.as<uint32_t>(),
                        h->ev[0], h->ev[1]);
  if (rc != BPPGPU_OK) return rc;
  float ms = 0;
  BPP_CUDA(cudaEventElapsedTime(&ms, h->ev[0], h->ev[1]));
  h->last_ms = ms;
  h->n_reps = n_replicates;
  return BPPGPU_OK;
}

int bppgpu_parsimony_score_replicates(bppgpu_parsimony* h, int32_t n_entries, const int32_t* rep, int32_t n_nodes, int32_t root,
                                      const int32_t* child_offsets, const int32_t* children, const int32_t* leaf_row, int64_t* score,
                                      uint32_t* site_scores) {
  if (!score || !rep) BPP_FAIL(BPPGPU_E_INVALID, "rep and score must not be NULL");
  return run(h, replicate_batch(h, n_entries, rep, n_nodes, root, child_offsets, children, leaf_row), false, nullptr, score, site_scores);
}

int bppgpu_parsimony_nni_replicates(bppgpu_parsimony* h, int32_t n_entries, const int32_t* rep, int32_t n_nodes, int32_t root,
                                    const int32_t* child_offsets, const int32_t* children, const int32_t* leaf_row, int64_t* delta,
                                    int64_t* score) {
  if (!delta || !rep) BPP_FAIL(BPPGPU_E_INVALID, "rep and delta must not be NULL");
  return run(h, replicate_batch(h, n_entries, rep, n_nodes, root, child_offsets, children, leaf_row), true, delta, score, nullptr);
}

int bppgpu_bootstrap_weights(int device, int64_t n_sites, const int64_t* indices, int64_t n_patterns, int64_t first_replicate,
                             int32_t n_replicates, uint64_t seed, uint32_t* weights) {
  if (!indices || !weights || n_patterns < 1) BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_bootstrap_weights");
  if (n_sites < 1 || n_sites >= ((int64_t)1 << 32)) BPP_FAIL(BPPGPU_E_INVALID, "n_sites must be in 1 .. 2^32 - 1, got %lld", (long long)n_sites);
  if (n_replicates < 1) BPP_FAIL(BPPGPU_E_INVALID, "n_replicates must be >= 1, got %d", n_replicates);
  int rc = check_device(device);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(cudaSetDevice(device));
  cudaStream_t st = nullptr;
  BPP_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
  std::unique_ptr<CUstream_st, cudaError_t (*)(cudaStream_t)> own(st, cudaStreamDestroy);
  DevBuf out;
  BPP_CUDA(out.ensure((size_t)n_replicates * n_patterns * 4));
  rc = draw_weights(device, st, n_sites, indices, n_patterns, first_replicate, n_replicates, seed, out.as<uint32_t>(), nullptr, nullptr);
  if (rc != BPPGPU_OK) return rc;
  BPP_CUDA(staged_copy(weights, out.p, (size_t)n_replicates * n_patterns * 4, false, device));
  return BPPGPU_OK;
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
