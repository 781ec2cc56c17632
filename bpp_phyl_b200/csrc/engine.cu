// libbppgpu: implementation of the C ABI in include/bppgpu.h (sm_100a only, no CPU fallback).
//
// Host planner: flattens the tree into a post-order walk program (Sethi-Ullman ordered so
// the on-chip CLV stack stays logarithmic), owns all device buffers, and enqueues
//   K1  pt_eigen_kernel / pt_series_kernel   P, r.P', r^2.P'' for every (point, branch, class)
//   K2b tiptab_kernel                         tip-code lookup tables
//   K2+K3 walk4 / walkS / generic             pruning + root reduction
//   K4+K5 upper / deriv kernels               prefix pass and branch derivatives
// on one stream; bppgpu_eval synchronises once at the end, bppgpu_eval_device not at all.
#include "engine.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <thread>

#include <dlfcn.h>
#include <nccl.h>   // declarations only: the library is dlopen()ed at bppgpu_comm_init, so libbppgpu has no link-time NCCL dependency

namespace bppgpu {

// NCCL entry points, resolved on first use.  In a process that already holds an NCCL (e.g. torch's bundled copy) dlopen by
// SONAME returns that one, so the engine and the host program share one NCCL runtime.
struct NcclApi {
  void* handle = nullptr;
  decltype(&ncclGetUniqueId) GetUniqueId = nullptr;
  decltype(&ncclCommInitRank) CommInitRank = nullptr;
  decltype(&ncclCommDestroy) CommDestroy = nullptr;
  decltype(&ncclAllReduce) AllReduce = nullptr;
  decltype(&ncclAllGather) AllGather = nullptr;
  decltype(&ncclGetErrorString) GetErrorString = nullptr;
  bool ok = false;
};
static NcclApi& nccl_api() {
  static NcclApi api;
  if (api.handle) return api;
  for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
    api.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
    if (api.handle) break;
  }
  if (!api.handle) return api;
  api.GetUniqueId = (decltype(api.GetUniqueId))dlsym(api.handle, "ncclGetUniqueId");
  api.CommInitRank = (decltype(api.CommInitRank))dlsym(api.handle, "ncclCommInitRank");
  api.CommDestroy = (decltype(api.CommDestroy))dlsym(api.handle, "ncclCommDestroy");
  api.AllReduce = (decltype(api.AllReduce))dlsym(api.handle, "ncclAllReduce");
  api.AllGather = (decltype(api.AllGather))dlsym(api.handle, "ncclAllGather");
  api.GetErrorString = (decltype(api.GetErrorString))dlsym(api.handle, "ncclGetErrorString");
  api.ok = api.GetUniqueId && api.CommInitRank && api.CommDestroy && api.AllReduce && api.AllGather && api.GetErrorString;
  return api;
}
#define BPP_NCCL(expr)                                                                                  \
  do {                                                                                                  \
    ncclResult_t _r = (expr);                                                                           \
    if (_r != ncclSuccess) BPP_FAIL(BPPGPU_E_NCCL, "NCCL error at %s:%d: %s", __FILE__, __LINE__, nccl_api().GetErrorString(_r)); \
  } while (0)

std::string& last_error() {
  static thread_local std::string s;
  return s;
}

static int g_sm_count = 148;
static int g_smem_per_sm = 228 * 1024;   // cudaDeviceProp::sharedMemPerMultiprocessor
static int g_smem_optin = 227 * 1024;    // cudaDeviceProp::sharedMemPerBlockOptin

template <typename T>
static cudaError_t dev_alloc(bppgpu_engine* e, T** p, size_t n) {
  *p = nullptr;
  if (n == 0) n = 1;
  cudaError_t r = cudaMalloc((void**)p, n * sizeof(T));
  if (r == cudaSuccess && e) e->bytes_resident += n * sizeof(T);
  return r;
}

static bool is_pow2(int v) { return v > 0 && (v & (v - 1)) == 0; }
static int ilog2(int v) {
  int l = 0;
  while ((1 << l) < v) ++l;
  return l;
}

// ---- walk program -----------------------------------------------------------------
// Children with the larger Sethi-Ullman label are evaluated first, so the number of
// live intermediate CLVs (stack slots) is minimal; the multiplication order inside an
// op stays the reference's son order (RHomogeneousTreeLikelihood.cpp:827-861).
// reg_slot (walk4c): a push whose lifetime contains no other push -- the sibling evaluated next has label 1, i.e. is a
// caterpillar -- goes to the kernel's register slot (dst_slot = -2, child kind CHILD_RSLOT) instead of a shared-memory slot.
// folded (walk4c): nodes the program treats as tips (CHILD_TIP, idx -1): cherries whose rows the table pass computes.
static void build_program(bppgpu_engine* e, Program& pr, bool all_keep, bool reg_slot = false,
                          const std::vector<char>* folded = nullptr) {
  const int nn = e->nn;
  auto is_leaf = [&](int n) { return e->leaf_slot[n] >= 0 || (folded && (*folded)[n]); };
  std::vector<int> label(nn, 0);
  // node ids are arbitrary: compute labels by an explicit post-order
  std::vector<int> order;
  order.reserve(nn);
  {
    std::vector<std::pair<int, int>> st;
    st.push_back({e->root, 0});
    while (!st.empty()) {
      auto& top = st.back();
      int n = top.first;
      int nc = e->child_off[n + 1] - e->child_off[n];
      if (top.second < nc) {
        int ch = e->children[e->child_off[n] + top.second];
        top.second++;
        st.push_back({ch, 0});
      } else {
        order.push_back(n);
        st.pop_back();
      }
    }
  }
  for (int n : order) {
    int nc = e->child_off[n + 1] - e->child_off[n];
    if (nc == 0) continue;
    std::vector<int> ls;
    for (int j = 0; j < nc; ++j) {
      int ch = e->children[e->child_off[n] + j];
      if (!is_leaf(ch)) ls.push_back(label[ch]);
    }
    std::sort(ls.begin(), ls.end(), std::greater<int>());
    int lab = 1;
    for (size_t i = 0; i < ls.size(); ++i) lab = std::max(lab, ls[i] + (int)i);
    label[n] = lab;
  }
  pr.ops.clear();
  pr.childs.clear();
  pr.nslots = 0;
  std::vector<int> free_slots;
  int next_slot = 0;
  std::vector<int> slot_of(nn, -1);
  std::vector<int> op_of(nn, -1);
  // iterative emission
  std::function<void(int)> emit = [&](int n) {
    int nc = e->child_off[n + 1] - e->child_off[n];
    std::vector<int> internal;
    for (int j = 0; j < nc; ++j) {
      int ch = e->children[e->child_off[n] + j];
      if (!is_leaf(ch)) internal.push_back(ch);
    }
    std::stable_sort(internal.begin(), internal.end(), [&](int a, int b) { return label[a] > label[b]; });
    for (size_t i = 0; i < internal.size(); ++i) {
      emit(internal[i]);
      if (!all_keep && reg_slot && i + 2 == internal.size() && label[internal[i + 1]] == 1) {
        slot_of[internal[i]] = -2;
        pr.ops[op_of[internal[i]]].dst_slot = -2;
      } else if (!all_keep && i + 1 < internal.size()) {
        int s;
        if (!free_slots.empty()) {
          s = free_slots.back();
          free_slots.pop_back();
        } else {
          s = next_slot++;
        }
        slot_of[internal[i]] = s;
        pr.ops[op_of[internal[i]]].dst_slot = s;
      }
    }
    Op op{};
    op.node = n;
    op.nchild = nc;
    op.child_begin = (int)pr.childs.size();
    op.dst_slot = -1;
    op.keep_idx = (e->keep || all_keep) ? e->internal_idx[n] : -1;
    op.is_root = n == e->root;
    for (int j = 0; j < nc; ++j) {
      int ch = e->children[e->child_off[n] + j];
      Child c{};
      c.pnode = ch;
      if (is_leaf(ch)) {
        c.kind = CHILD_TIP;
        c.idx = e->leaf_slot[ch];
      } else if (all_keep) {
        c.kind = CHILD_KEEP;
        c.idx = e->internal_idx[ch];
      } else if (slot_of[ch] >= 0) {
        c.kind = CHILD_SLOT;
        c.idx = slot_of[ch];
      } else if (slot_of[ch] == -2) {
        c.kind = CHILD_RSLOT;
        c.idx = 0;
      } else {
        c.kind = CHILD_REG;
        c.idx = 0;
      }
      pr.childs.push_back(c);
    }
    for (int ch : internal) {
      if (slot_of[ch] >= 0) free_slots.push_back(slot_of[ch]);
      slot_of[ch] = -1;
    }
    op_of[n] = (int)pr.ops.size();
    pr.ops.push_back(op);
  };
  if (e->leaf_slot[e->root] < 0) emit(e->root);
  pr.nslots = next_slot;
}

static int upload_program(bppgpu_engine* e, Program& pr) {
  BPP_CUDA(dev_alloc(e, &pr.d_ops, pr.ops.size()));
  BPP_CUDA(dev_alloc(e, &pr.d_childs, pr.childs.size()));
  if (!pr.ops.empty())
    BPP_CUDA(cudaMemcpy(pr.d_ops, pr.ops.data(), pr.ops.size() * sizeof(Op), cudaMemcpyHostToDevice));
  if (!pr.childs.empty())
    BPP_CUDA(cudaMemcpy(pr.d_childs, pr.childs.data(), pr.childs.size() * sizeof(Child), cudaMemcpyHostToDevice));
  return BPPGPU_OK;
}

static int check_device(int device) {
  int n = 0;
  cudaError_t r = cudaGetDeviceCount(&n);
  if (r != cudaSuccess || n == 0)
    BPP_FAIL(BPPGPU_E_CUDA, "no usable CUDA device (%s); libbppgpu has no CPU fallback",
             r == cudaSuccess ? "device count is 0" : cudaGetErrorString(r));
  if (device < 0 || device >= n) BPP_FAIL(BPPGPU_E_INVALID, "device %d out of range (0..%d)", device, n - 1);
  BPP_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  BPP_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major < 10) BPP_FAIL(BPPGPU_E_CUDA, "device %d is sm_%d%d; libbppgpu is built for sm_100a only", device, prop.major, prop.minor);
  g_sm_count = prop.multiProcessorCount;
  g_smem_per_sm = (int)prop.sharedMemPerMultiprocessor;
  g_smem_optin = (int)prop.sharedMemPerBlockOptin;
  // dynamic shared memory above 48 KB is opt-in
  BPP_CUDA(cudaFuncSetAttribute(pt_dmma_kernel<8, 1, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(pt_dmma_kernel<8, 2, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(pt_dmma_kernel<8, 4, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(pt_dmma_stacked_kernel<8, 4, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_node_kernel<5, 3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_node_kernel<16, 8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_node_kernel<16, 8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_node_kernel<5, 3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_node_kernel<5, 3, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_upper_deriv_kernel<5, 3, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_upper_deriv_kernel<5, 3, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  BPP_CUDA(cudaFuncSetAttribute(dmma_upper_deriv_kernel<16, 8, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  return BPPGPU_OK;
}

// ---- programmatic dependent launch of the per-node kernels (common.cuh: pdl_wait / pdl_launch_dependents) -------------------
// `overlap` = this launch may start while its predecessor in the stream drains.  The first per-node launch of a pass is launched
// plainly: what precedes it (operand packing) must be complete before any CTA of the chain stages operands.
static const bool g_pdl_on = getenv("BPPGPU_PDL") && atoi(getenv("BPPGPU_PDL")) != 0;   // opt-in: measured, no gain (DESIGN 3.3)
template <typename P>
static cudaError_t launch_node_kernel(void (*kern)(P), unsigned grid, unsigned threads, size_t smem, cudaStream_t st, bool overlap,
                                      const P& params) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = (overlap && g_pdl_on) ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kern, params);
}

// ---- model upload -------------------------------------------------------------------
static void free_model(DevModel& m) {
  cudaFree(m.slab);
  cudaFree(m.pslab);
  m = DevModel{};
}

// Host-side image of a model slab: [V | Vinv | re | im | role(int) | pad] [Q | Q2].  The head is all an eigen-route model without
// generator needs, so it travels alone (half the bytes of a batched-points upload).
static size_t model_head_doubles(int S) { return (((size_t)2 * S * S + 2 * (size_t)S + ((size_t)S + 1) / 2) + 31) & ~(size_t)31; }
static size_t model_slab_doubles(int S) { return model_head_doubles(S) + (size_t)2 * S * S; }

// pslab of a model = [Vp | Vinvp | rep | imp], the copies the tensor-core P(t) kernel reads when S is not a multiple of 8 or the
// spectrum has conjugate pairs: zero-padded to Sp, eigen-columns permuted so that every pair starts at an even index (pairs first,
// then the real eigenvalues).  Built on the device from the slab that has just arrived: no second host image, no second copy.
__global__ void model_permute_kernel(const double* __restrict__ V, const double* __restrict__ Vinv, const double* __restrict__ re,
                                     const double* __restrict__ im, const int* __restrict__ role, int S, int Sp, double* __restrict__ pslab) {
  __shared__ int order[256];
  if (threadIdx.x == 0) {
    int n = 0;
    for (int k = 0; k < S; ++k)
      if (role[k] == 1) { order[n++] = k; order[n++] = k + 1; }
    for (int k = 0; k < S; ++k)
      if (role[k] == 0) order[n++] = k;
  }
  __syncthreads();
  double *vp = pslab, *vip = vp + (size_t)Sp * Sp, *rp = vip + (size_t)Sp * Sp, *ip = rp + Sp;
  for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < Sp * Sp; idx += gridDim.x * blockDim.x) {
    const int i = idx / Sp, j = idx - i * Sp;
    vp[idx] = (i < S && j < S) ? V[(size_t)i * S + order[j]] : 0.0;     // vp[i][j]   = V[i][order[j]]
    vip[idx] = (i < S && j < S) ? Vinv[(size_t)order[i] * S + j] : 0.0; // vip[i][j]  = Vinv[order[i]][j]
  }
  if (blockIdx.x == 0)
    for (int j = threadIdx.x; j < Sp; j += blockDim.x) {
      rp[j] = j < S ? re[order[j]] : 0.0;
      ip[j] = j < S ? im[order[j]] : 0.0;
    }
}

// Fills `img` (host, model_slab_doubles(S) doubles; only the first *used are written and need to travel) from the descriptor and
// the scalar fields of dm; *padded = the tensor-core kernel needs the permuted copies.  No CUDA call: set_models stages many images.
static int build_model_image(DevModel& dm, const bppgpu_model_desc* m, int S, bool need_q2, bool keep_q, double* img, size_t* used, bool* padded) {
  const size_t SS = (size_t)S * S, head = model_head_doubles(S);
  const bool eigen = (m->flags & BPPGPU_MODEL_NONSINGULAR) != 0;
  if (eigen && (!m->right_eigen || !m->left_eigen || !m->eigen_re))
    BPP_FAIL(BPPGPU_E_INVALID, "model flagged NONSINGULAR needs right_eigen, left_eigen and eigen_re");
  if (!eigen && !m->generator) BPP_FAIL(BPPGPU_E_INVALID, "singular model needs its generator");
  if ((m->flags & BPPGPU_MODEL_CHR_DERIV) && !m->generator) BPP_FAIL(BPPGPU_E_INVALID, "BPPGPU_MODEL_CHR_DERIV needs the generator");
  dm.flags = m->flags;
  dm.rate = m->rate;
  dm.eps = m->taylor_epsilon > 0 ? m->taylor_epsilon : 1e-4;
  dm.has_complex = 0;
  // the generator only travels when a route of this model reads it: series (singular), the Chromosome derivative forms, exact expm
  const bool want_q = m->generator && (keep_q || !eigen || (m->flags & (BPPGPU_MODEL_CHR_DERIV | BPPGPU_MODEL_CHR_TAYLOR | BPPGPU_MODEL_EXACT_EXPM)));
  dm.has_Q = want_q;
  dm.q_l1 = 0.0;
  double *iV = img, *iVinv = img + SS, *ire = img + 2 * SS, *iim = ire + S, *iQ = img + head, *iQ2 = iQ + SS;
  int* irole = reinterpret_cast<int*>(iim + S);
  *used = want_q ? model_slab_doubles(S) : head;
  if (eigen) {
    memcpy(iV, m->right_eigen, SS * 8);
    memcpy(iVinv, m->left_eigen, SS * 8);
    memcpy(ire, m->eigen_re, S * 8);
    std::fill(iim, img + head, 0.0);   // im, role, pad
    if (m->eigen_im) {
      memcpy(iim, m->eigen_im, S * 8);
      // conjugate pairs are adjacent, the +im member first (JAMA EigenValue convention,
      // AbstractSubstitutionModel.cpp:438-468 walks them the same way)
      for (int k = 0; k < S; ++k) {
        if (iim[k] != 0.0 && irole[k] == 0) {
          if (k + 1 >= S || iim[k + 1] == 0.0) BPP_FAIL(BPPGPU_E_INVALID, "unpaired complex eigenvalue at index %d", k);
          irole[k] = 1;
          irole[k + 1] = 2;
          dm.has_complex = 1;
        }
      }
    }
  } else {
    std::fill(img, img + head, 0.0);
  }
  const int Sp = (S + 7) & ~7;
  *padded = eigen && S >= 32 && Sp <= 256 && (Sp != S || dm.has_complex);   // the sizes the tensor-core P(t) kernel takes
  if (want_q) {
    memcpy(iQ, m->generator, SS * 8);
    std::fill(iQ2, iQ2 + SS, 0.0);
    double l1 = 0.0;
    for (size_t i = 0; i < SS; ++i) l1 += std::fabs(m->generator[i]);
    dm.q_l1 = l1;
    if (need_q2 && ((m->flags & BPPGPU_MODEL_CHR_DERIV) || !eigen))   // Q.Q for the Chromosome second derivative (Q^2.P)
      for (int i = 0; i < S; ++i)
        for (int k = 0; k < S; ++k) {
          const double a = m->generator[(size_t)i * S + k];
          if (a == 0.0) continue;
          for (int j = 0; j < S; ++j) iQ2[(size_t)i * S + j] += a * m->generator[(size_t)k * S + j];
        }
  }
  return BPPGPU_OK;
}

// device storage of a model slot (first upload, or a change of shape) and the pointers into it
static int ensure_model_storage(DevModel& dm, int S, bool padded) {
  const size_t SS = (size_t)S * S;
  if (!dm.slab || dm.S != S) {   // (only the storage: the scalar fields were just filled by build_model_image)
    cudaFree(dm.slab);
    cudaFree(dm.pslab);
    dm.slab = dm.pslab = nullptr;
    BPP_CUDA(cudaMalloc(&dm.slab, model_slab_doubles(S) * 8));
    dm.S = S;
  }
  dm.V = dm.slab; dm.Vinv = dm.slab + SS;
  dm.re = dm.slab + 2 * SS; dm.im = dm.re + S;
  dm.role = reinterpret_cast<int*>(dm.im + S);
  dm.Q = dm.slab + model_head_doubles(S); dm.Q2 = dm.Q + SS;
  const int Sp = (S + 7) & ~7;
  if (padded) {
    if (!dm.pslab) BPP_CUDA(cudaMalloc(&dm.pslab, ((size_t)2 * Sp * Sp + 2 * Sp) * 8));
    dm.Vp = dm.pslab; dm.Vinvp = dm.pslab + (size_t)Sp * Sp; dm.rep = dm.Vinvp + (size_t)Sp * Sp; dm.imp = dm.rep + Sp;
  } else if (Sp == S) {
    dm.Vp = dm.V; dm.Vinvp = dm.Vinv; dm.rep = dm.re; dm.imp = dm.im;
  } else {
    dm.Vp = dm.Vinvp = dm.rep = dm.imp = nullptr;   // S < 32 and not a multiple of 8: the CUDA-core P(t) kernel reads V .. re
  }
  return BPPGPU_OK;
}

// the image -> the slot's slab on `st`, then the permuted copies from it (stream order)
static int send_model_image(DevModel& dm, int S, const double* img, size_t used, bool padded, cudaStream_t st) {
  BPP_CUDA(cudaMemcpyAsync(dm.slab, img, used * 8, cudaMemcpyHostToDevice, st));
  if (padded) {
    const int Sp = (S + 7) & ~7;
    model_permute_kernel<<<std::min(64, (Sp * Sp + 255) / 256), 256, 0, st>>>(dm.V, dm.Vinv, dm.re, dm.im, dm.role, S, Sp, dm.pslab);
    BPP_CUDA(cudaGetLastError());
  }
  return BPPGPU_OK;
}

static int upload_model(DevModel& dm, const bppgpu_model_desc* m, int S, bool need_q2 = true) {
  std::vector<double> img(model_slab_doubles(S));
  size_t used = 0;
  bool padded = false;
  int rc = build_model_image(dm, m, S, need_q2, /*keep_q=*/need_q2, img.data(), &used, &padded);
  if (rc) return rc;
  rc = ensure_model_storage(dm, S, padded);
  if (rc) return rc;
  rc = send_model_image(dm, S, img.data(), used, padded, 0);
  if (rc) return rc;
  BPP_CUDA(cudaStreamSynchronize(0));   // img goes out of scope
  dm.set = true;
  return BPPGPU_OK;
}

static ModelDev to_dev(const DevModel& m) {
  ModelDev d{};
  d.V = m.V; d.Vinv = m.Vinv; d.re = m.re; d.im = m.im; d.role = m.role; d.Q = m.has_Q ? m.Q : nullptr; d.Q2 = m.has_Q ? m.Q2 : nullptr;
  d.Vp = m.Vp; d.Vinvp = m.Vinvp; d.rep = m.rep; d.imp = m.imp;
  d.rate = m.rate; d.eps = m.eps; d.q_l1 = m.q_l1; d.flags = m.flags; d.has_complex = m.has_complex;
  return d;
}

// enqueue K1 for `npts` points starting at `p0` (tables indexed from 0 within the chunk)
static int launch_pt(cudaStream_t st, const ModelDev* d_models, bool any_series, bool any_chr_deriv, bool any_real_eigen,
                     bool any_complex, bool stacked_ok,
                     const int* d_branch_model, const double* d_brlen, const double* d_rates, int S, int C,
                     int nn, int root, int npts, unsigned want, double* P, double* dP, double* d2P,
                     double* scratch, int* d_status, long long* launches) {
  PtParams pp{};
  pp.models = d_models;
  pp.branch_model = d_branch_model;
  pp.brlen = d_brlen;
  pp.rates = d_rates;
  pp.S = S; pp.C = C; pp.nn = nn; pp.root = root;
  pp.want = want;
  pp.P = P; pp.dP = dP; pp.d2P = d2P;
  pp.Pun = any_chr_deriv && (want & 6u) ? scratch : nullptr;
  const int nmat = npts * nn * C;
  if (nmat == 0) return BPPGPU_OK;
  const int threads = S * S >= 256 ? 256 : (S * S >= 64 ? 64 : 32);
  const int Sp = (S + 7) & ~7;
  pp.dmma_real = 0;
  if (S >= 32 && Sp <= 256 && (any_real_eigen || any_complex)) {
    // FP64 tensor-core GEMM for every eigen-path matrix (real spectra and conjugate-pair block form)
    pp.dmma_real = 1;
    const int nblk = Sp / 8;
    if (stacked_ok && nblk > 16 && nblk * 1 >= 6 && !any_series) {
      // one model per point: stack the row blocks of the point's matrices (perfect balance, see pt_dmma_kernels.cuh)
      constexpr int RB = 32;
      const long long total_rb = (long long)nn * C * nblk;
      const dim3 grid((unsigned)((total_rb + RB - 1) / RB), (unsigned)((nblk + 4) / 5), (unsigned)npts);
      pt_dmma_stacked_kernel<8, 4, 5><<<grid, 256, pt_dmma_stacked_smem_bytes(Sp, 5), st>>>(pp, Sp);
    } else if (nblk <= 8) {
      pt_dmma_kernel<8, 1, 8><<<dim3(nmat, 1), 256, pt_dmma_smem_bytes(Sp, 8), st>>>(pp, Sp);
    } else if (nblk <= 16) {
      pt_dmma_kernel<8, 2, 8><<<dim3(nmat, (nblk + 7) / 8), 256, pt_dmma_smem_bytes(Sp, 8), st>>>(pp, Sp);
    } else {
      pt_dmma_kernel<8, 4, 5><<<dim3(nmat, (nblk + 4) / 5), 256, pt_dmma_smem_bytes(Sp, 5), st>>>(pp, Sp);
    }
    ++*launches;
  }
  if (!pp.dmma_real) {
    pt_eigen_kernel<<<nmat, threads, 6 * S * sizeof(double), st>>>(pp);
    ++*launches;
  }
  if (any_chr_deriv && (want & 6u)) {
    SeriesParams sp{};
    sp.pt = pp;
    sp.scratch = scratch;
    sp.status = d_status;
    pt_chr_deriv_kernel<<<nmat, threads, 0, st>>>(sp);
    ++*launches;
  }
  if (any_series) {
    SeriesParams sp{};
    sp.pt = pp;
    sp.scratch = scratch;
    sp.status = d_status;
    static const int sparse_env = getenv("BPPGPU_SERIES_SPARSE") ? atoi(getenv("BPPGPU_SERIES_SPARSE")) : 0;
    sp.sparse_terms = sparse_env;
    if (S >= 32 && S <= 8 * kChrWarps * kChrMaxRB) {   // matrix products on the FP64 tensor cores
      const size_t smem = (size_t)((S + 7) & ~7) * kChrLD * sizeof(double) + sparse_cols_bytes(S);   // B panel + compressed columns of Q
      BPP_CUDA(cudaFuncSetAttribute(pt_series_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
      pt_series_kernel<true><<<nmat, kChrWarps * 32, smem, st>>>(sp);
    } else {
      pt_series_kernel<false><<<nmat, threads, 0, st>>>(sp);
    }
    ++*launches;
  }
  BPP_CUDA(cudaGetLastError());
  return BPPGPU_OK;
}

}  // namespace bppgpu

using namespace bppgpu;

// =====================================================================================
// (C linkage comes from the declarations in include/bppgpu.h)

const char* bppgpu_last_error(void) { return last_error().c_str(); }
int bppgpu_abi_version(void) { return 2; }
int bppgpu_sizeof(int which) {
  switch (which) {
    case 0: return (int)sizeof(bppgpu_model_desc);
    case 1: return (int)sizeof(bppgpu_config);
    case 2: return (int)sizeof(bppgpu_stats);
    default: return -1;
  }
}

int bppgpu_device_count(int* n) {
  if (!n) BPP_FAIL(BPPGPU_E_INVALID, "null argument");
  int c = 0;
  cudaError_t r = cudaGetDeviceCount(&c);
  if (r != cudaSuccess) {
    *n = 0;
    cudaGetLastError();
    return BPPGPU_OK;
  }
  *n = c;
  return BPPGPU_OK;
}

// ---- site patterns (host) ---------------------------------------------------------------
int bppgpu_site_patterns(const uint8_t* columns, int64_t n_sites, int32_t col_bytes, int64_t* pattern_site,
                         uint32_t* weights, int64_t* indices, int64_t* n_patterns) {
  if (n_sites < 0 || col_bytes <= 0 || !n_patterns || (n_sites > 0 && (!columns || !pattern_site || !weights || !indices)))
    BPP_FAIL(BPPGPU_E_INVALID, "bad argument to bppgpu_site_patterns");
  *n_patterns = 0;
  if (n_sites == 0) return BPPGPU_OK;
  std::vector<int64_t> order((size_t)n_sites);
  for (int64_t i = 0; i < n_sites; ++i) order[(size_t)i] = i;
  const size_t w = (size_t)col_bytes;
  // std::sort like the reference; ties are identical columns, so their relative order cannot change the result
  // except for WHICH identical site represents the pattern -- we take the smallest original position
  std::sort(order.begin(), order.end(), [&](int64_t a, int64_t b) {
    const int c = memcmp(columns + (size_t)a * w, columns + (size_t)b * w, w);
    return c != 0 ? c < 0 : a < b;
  });
  int64_t np = 0;
  pattern_site[0] = order[0];
  weights[0] = 1;
  indices[order[0]] = 0;
  for (int64_t k = 1; k < n_sites; ++k) {
    const int64_t cur = order[(size_t)k], prev = order[(size_t)k - 1];
    if (memcmp(columns + (size_t)cur * w, columns + (size_t)prev * w, w) == 0) {
      weights[np]++;
    } else {
      ++np;
      pattern_site[np] = cur;
      weights[np] = 1;
    }
    indices[cur] = np;
  }
  *n_patterns = np + 1;
  return BPPGPU_OK;
}

// ---- Interface 1 ----------------------------------------------------------------------
int bppgpu_pt_batch(int device, const bppgpu_model_desc* model, int64_t n_t, const double* t, unsigned want,
                    double* P, double* dP, double* d2P) {
  if (!model || !t || n_t < 0) BPP_FAIL(BPPGPU_E_INVALID, "null model / t or negative n_t");
  const int S = model->n_states;
  if (S <= 0) BPP_FAIL(BPPGPU_E_INVALID, "n_states must be positive");
  if (((want & 1u) && !P) || ((want & 2u) && !dP) || ((want & 4u) && !d2P))
    BPP_FAIL(BPPGPU_E_INVALID, "output pointer missing for a requested table");
  int rc = check_device(device);
  if (rc) return rc;
  if (n_t == 0) return BPPGPU_OK;
  DevModel dm;
  rc = upload_model(dm, model, S);
  if (rc) { free_model(dm); return rc; }
  ModelDev md = to_dev(dm);
  const size_t SS = (size_t)S * S;
  ModelDev* d_md = nullptr;
  int* d_bm = nullptr;
  double *d_t = nullptr, *d_r = nullptr, *dPm = nullptr, *ddP = nullptr, *dd2P = nullptr, *scr = nullptr;
  int* d_status = nullptr;
  const bool series = !(model->flags & BPPGPU_MODEL_NONSINGULAR);
  const bool chrd = (model->flags & BPPGPU_MODEL_CHR_DERIV) && !series;
  auto cleanup = [&]() {
    cudaFree(d_md); cudaFree(d_bm); cudaFree(d_t); cudaFree(d_r); cudaFree(dPm); cudaFree(ddP); cudaFree(dd2P);
    cudaFree(scr); cudaFree(d_status);
    free_model(dm);
  };
#define PT_CUDA(x)                                                                      \
  do {                                                                                  \
    cudaError_t _e = (x);                                                               \
    if (_e != cudaSuccess) {                                                            \
      cleanup();                                                                        \
      BPP_FAIL(_e == cudaErrorMemoryAllocation ? BPPGPU_E_NOMEM : BPPGPU_E_CUDA, "CUDA error %s at %s:%d: %s", \
               cudaGetErrorName(_e), __FILE__, __LINE__, cudaGetErrorString(_e));      \
    }                                                                                   \
  } while (0)
  PT_CUDA(cudaMalloc(&d_md, sizeof(ModelDev)));
  PT_CUDA(cudaMemcpy(d_md, &md, sizeof(ModelDev), cudaMemcpyHostToDevice));
  PT_CUDA(cudaMalloc(&d_bm, n_t * sizeof(int)));
  PT_CUDA(cudaMemset(d_bm, 0, n_t * sizeof(int)));
  PT_CUDA(cudaMalloc(&d_t, n_t * 8));
  PT_CUDA(cudaMemcpy(d_t, t, n_t * 8, cudaMemcpyHostToDevice));
  const double one = 1.0;
  PT_CUDA(cudaMalloc(&d_r, 8));
  PT_CUDA(cudaMemcpy(d_r, &one, 8, cudaMemcpyHostToDevice));
  PT_CUDA(cudaMalloc(&d_status, 4));
  PT_CUDA(cudaMemset(d_status, 0, 4));
  if (want & 1u) PT_CUDA(cudaMalloc(&dPm, n_t * SS * 8));
  if (want & 2u) PT_CUDA(cudaMalloc(&ddP, n_t * SS * 8));
  if (want & 4u) PT_CUDA(cudaMalloc(&dd2P, n_t * SS * 8));
  if (series) PT_CUDA(cudaMalloc(&scr, n_t * 4 * SS * 8));
  else if (chrd) PT_CUDA(cudaMalloc(&scr, n_t * SS * 8));
  long long launches = 0;
  rc = launch_pt(nullptr, d_md, series, chrd, !series && !dm.has_complex, !series && dm.has_complex, false, d_bm, d_t, d_r, S, 1,
                 (int)n_t, -1, 1, want, dPm, ddP, dd2P, scr, d_status, &launches);
  if (rc) { cleanup(); return rc; }
  PT_CUDA(cudaDeviceSynchronize());
  if (want & 1u) PT_CUDA(cudaMemcpy(P, dPm, n_t * SS * 8, cudaMemcpyDeviceToHost));
  if (want & 2u) PT_CUDA(cudaMemcpy(dP, ddP, n_t * SS * 8, cudaMemcpyDeviceToHost));
  if (want & 4u) PT_CUDA(cudaMemcpy(d2P, dd2P, n_t * SS * 8, cudaMemcpyDeviceToHost));
  int status = 0;
  PT_CUDA(cudaMemcpy(&status, d_status, 4, cudaMemcpyDeviceToHost));
  cleanup();
#undef PT_CUDA
  if (status) BPP_FAIL(BPPGPU_E_NUMERIC, "ChromosomeSubstitutionModel: Taylor series did not reach convergence!");
  return BPPGPU_OK;
}

// ---- Interface 2 ----------------------------------------------------------------------
int bppgpu_destroy(bppgpu_engine* e) {
  if (!e) return BPPGPU_OK;
  cudaSetDevice(e->dev);
  if (e->stream) cudaStreamSynchronize(e->stream);
  void* ptrs[] = {e->d_codes, e->d_code_table, e->d_code_single, e->d_weights, e->d_rates, e->d_probs, e->d_rootfreq,
                  e->d_rootfreq_used, e->d_brlen, e->d_branch_model, e->d_leaf_nodes, e->d_models, e->d_P, e->d_dP,
                  e->d_d2P, e->d_tiptab, e->d_keep, e->d_keep_exp, e->d_gstack, e->d_gstack_exp, e->d_upper,
                  e->d_upper_exp, e->d_SR, e->d_rexp, e->d_site_lnl, e->d_partials, e->d_partials2, e->d_out,
                  e->prog.d_ops, e->prog.d_childs, e->gprog.d_ops, e->gprog.d_childs, e->d_sibs, e->d_scratch,
                  e->d_dtiptab, e->d_d2tiptab, e->d_dLc, e->d_fam_mask, e->d_fam_part, e->d_fam_packA, e->d_fam_packS, e->d_fam_packL, e->d_fam_packT, e->d_w4c_stream, e->d_w4c_blocks, e->d_w4c_tip_order, e->d_codesC, e->d_w4c_counter, e->d_w4_desc, e->d_w4_tip_order, e->d_w4_blocks, e->d_w4_stream, e->d_codesT,
                  e->d_status, e->d_wr_recs, e->d_chr_tile_edges, e->d_chr_tile_kind, e->d_chr_leaf_state, e->d_child_off,
                  e->d_children, e->d_chr_leaf_vec, e->d_chr_term, e->d_chr_term_exp, e->d_chr_bad, e->d_chr_guardP, e->d_chr_aslab, e->d_prune_nodes, e->d_family_nodes, e->d_chr_probe_t,
                  e->d_chr_probe_bm, e->d_models_noclamp, e->d_bad_idx, e->d_bad_brlen, e->d_bad_rootfreq, e->d_bad_rootfreq_used,
                  e->d_bad_site_lnl, e->d_bad_out, e->d_bad_branch_model};
  for (void* p : ptrs) cudaFree(p);
  for (auto& m : e->models) free_model(m);
  if (e->h_stage) cudaFreeHost(e->h_stage);
  for (int t = 0; t < bppgpu_engine::kStageThreads; ++t) {
    if (e->stage_stream[t]) cudaStreamDestroy(e->stage_stream[t]);
    for (int b = 0; b < 2; ++b)
      if (e->stage_ev[t][b]) cudaEventDestroy(e->stage_ev[t][b]);
  }
  if (e->comm && nccl_api().ok) nccl_api().CommDestroy((ncclComm_t)e->comm);
  e->comm = nullptr;
  if (e->eval_done) cudaEventDestroy(e->eval_done);
  if (e->ev0) cudaEventDestroy(e->ev0);
  if (e->ev1) cudaEventDestroy(e->ev1);
  for (int i = 0; i < bppgpu_engine::kRing; ++i) {
    if (e->ring_a[i]) cudaEventDestroy(e->ring_a[i]);
    if (e->ring_b[i]) cudaEventDestroy(e->ring_b[i]);
    if (e->ptring_a[i]) cudaEventDestroy(e->ptring_a[i]);
    if (e->ptring_b[i]) cudaEventDestroy(e->ptring_b[i]);
  }
  if (e->stream) cudaStreamDestroy(e->stream);
  delete e;
  return BPPGPU_OK;
}

static int walk4_dispatch(bppgpu_engine* e, const Walk4Params* wp, int grid, size_t, cudaStream_t st, bool attr_only);
static int walk4c_dispatch(bppgpu_engine* e, int pt, const Walk4cParams* wp, int grid, size_t smem, cudaStream_t st, bool attr_only);

static int create_impl(const bppgpu_config* cfg, bppgpu_engine* e) {
  e->dev = cfg->device;
  e->S = cfg->n_states; e->C = cfg->n_cats; e->N = cfg->n_patterns; e->nn = cfg->n_nodes; e->root = cfg->root;
  e->npoints = cfg->n_points; e->nmodels = cfg->n_models; e->ncodes = cfg->n_codes; e->code_bytes = cfg->code_bytes;
  e->flags = cfg->flags;
  e->keep = (cfg->flags & BPPGPU_FLAG_KEEP_CLVS) != 0;
  const int nn = e->nn, S = e->S, C = e->C;
  const long long N = e->N;
  e->child_off.assign(cfg->child_offsets, cfg->child_offsets + nn + 1);
  if (e->child_off[0] != 0) BPP_FAIL(BPPGPU_E_INVALID, "child_offsets[0] must be 0");
  for (int i = 0; i < nn; ++i)
    if (e->child_off[i + 1] < e->child_off[i]) BPP_FAIL(BPPGPU_E_INVALID, "child_offsets must be non-decreasing");
  e->children.assign(cfg->children, cfg->children + e->child_off[nn]);
  e->parent.assign(nn, -1);
  for (int n = 0; n < nn; ++n)
    for (int k = e->child_off[n]; k < e->child_off[n + 1]; ++k) {
      int ch = e->children[k];
      if (ch < 0 || ch >= nn || ch == e->root) BPP_FAIL(BPPGPU_E_INVALID, "bad child id %d of node %d", ch, n);
      if (e->parent[ch] != -1) BPP_FAIL(BPPGPU_E_INVALID, "node %d has two fathers", ch);
      e->parent[ch] = n;
    }
  for (int n = 0; n < nn; ++n)
    if (n != e->root && e->parent[n] < 0) BPP_FAIL(BPPGPU_E_INVALID, "node %d is not connected to the root", n);
  e->leaf_slot.assign(nn, -1);
  e->internal_idx.assign(nn, -1);
  for (int n = 0; n < nn; ++n) {
    if (e->child_off[n + 1] == e->child_off[n]) {
      e->leaf_slot[n] = e->nl++;
      e->leaf_nodes.push_back(n);
    } else {
      e->internal_idx[n] = e->ni++;
    }
  }
  if (e->leaf_slot[e->root] >= 0) BPP_FAIL(BPPGPU_E_INVALID, "the root must have sons");
  // pre-order (fathers first), cycle check
  {
    std::vector<int> st{e->root};
    while (!st.empty()) {
      int n = st.back();
      st.pop_back();
      e->preorder.push_back(n);
      for (int k = e->child_off[n + 1] - 1; k >= e->child_off[n]; --k) st.push_back(e->children[k]);
    }
    if ((int)e->preorder.size() != nn) BPP_FAIL(BPPGPU_E_INVALID, "topology is not a tree");
  }
  BPP_CUDA(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
  BPP_CUDA(cudaEventCreate(&e->ev0));
  BPP_CUDA(cudaEventCreate(&e->ev1));
  for (int i = 0; i < bppgpu_engine::kRing; ++i) {
    BPP_CUDA(cudaEventCreate(&e->ring_a[i]));
    BPP_CUDA(cudaEventCreate(&e->ring_b[i]));
    BPP_CUDA(cudaEventCreate(&e->ptring_a[i]));
    BPP_CUDA(cudaEventCreate(&e->ptring_b[i]));
  }

  // ---- path selection ---------------------------------------------------------------
  build_program(e, e->prog, false);
  // keep-buffer index of an internal node = its position in the walk (so the walk streams node o to slab o)
  for (size_t o = 0; o < e->prog.ops.size(); ++o) e->internal_idx[e->prog.ops[o].node] = (int)o;
  const bool cpow = is_pow2(C) && C <= 8;
  bool w4ok = S == 4 && cpow && e->code_bytes == 1 && e->prog.nslots <= 63 &&
              (size_t)e->prog.nslots * kWalk4Threads * 36 <= 200 * 1024;
  for (const Op& op : e->prog.ops)
    if (op.nchild > 6) w4ok = false;
  const bool wroot = (cfg->flags & BPPGPU_FLAG_WEIGHTED_ROOT) != 0;  // needs the root CLV in HBM: node-kernel paths
  if (wroot) w4ok = false;
  if (w4ok) e->path = PATH_WALK4;
  else e->path = PATH_GENERIC;
  // S = 20 register walk (walkS_kernel): measured 77 ms vs 41 ms for the tensor-core node kernels on the 500-taxon x 200k
  // config, so it is no longer a default; BPPGPU_PATH=walk selects it (value-only, no weighted root)
  const bool walks_ok = S == 20 && cpow && !e->keep && !wroot;
  (void)walks_ok;
  if (e->path == PATH_GENERIC && S % 4 == 0 && ((S > 16 && S <= 20) || (S > 56 && S <= 64))) e->path = PATH_DMMA;
  if (const char* env = getenv("BPPGPU_PATH")) {  // tuning knob
    if (!strcmp(env, "generic")) e->path = PATH_GENERIC;
    if (!strcmp(env, "walk") && walks_ok) e->path = PATH_WALKS;
    if (!strcmp(env, "dmma") && S % 4 == 0 && ((S > 16 && S <= 20) || (S > 56 && S <= 64))) e->path = PATH_DMMA;
  }
  if (cfg->flags & BPPGPU_FLAG_FORCE_GENERIC) e->path = PATH_GENERIC;
  // many parameter points on few patterns (ChromEvol): one launch per node covers every point of a chunk
  if (e->npoints > 1 && N * C <= 64 && !(cfg->flags & BPPGPU_FLAG_FORCE_GENERIC)) e->path = PATH_POINTS;
  if (e->path == PATH_GENERIC || e->path == PATH_DMMA || e->path == PATH_POINTS) e->keep = true;
  build_program(e, e->prog, false);  // again: keep indices are known now
  build_program(e, e->gprog, true);
  if (e->path == PATH_WALK4) {
    // packed descriptors, tip consumption order and table blocks, all in walk order
    size_t off = 0;
    for (const Op& op : e->prog.ops) {
      int shape = 0;
      if (op.nchild == 2) {
        const int ka = walk4_kind_index(e->prog.childs[op.child_begin].kind);
        const int kb = walk4_kind_index(e->prog.childs[op.child_begin + 1].kind);
        shape = 1 + 3 * ka + kb;
        if (shape == 5 || shape == 9) shape = 0;  // (SLOT,SLOT) / (REG,REG) cannot come out of the planner
      }
      unsigned long long d = (unsigned long long)shape | ((unsigned long long)op.nchild << 4) |
                             ((unsigned long long)(op.dst_slot + 1) << 8);
      for (int j = 0; j < op.nchild; ++j) {
        const Child& ch = e->prog.childs[op.child_begin + j];
        const unsigned tok = ((unsigned)ch.kind << 6) | (ch.kind == CHILD_SLOT ? (unsigned)ch.idx : 0u);
        d |= (unsigned long long)tok << (16 + 8 * j);
        PackBlock b{};
        b.kind = ch.kind;
        b.pnode = ch.pnode;
        b.off = (long long)off;
        e->w4_blocks.push_back(b);
        if (ch.kind == CHILD_TIP) {
          e->w4_tip_order.push_back(ch.idx);
          off += (size_t)e->ncodes * C * 4;
        } else {
          off += (size_t)C * 16;
        }
      }
      e->w4_desc.push_back(d);
    }
    e->w4_desc.push_back(0ull);  // sentinels read by the one-op-ahead prefetch
    e->w4_desc.push_back(0ull);
    e->w4_stream_len = off;
    e->w4_tstride = (int)(((e->w4_tip_order.size() + 7) / 8) * 8 + 16);
  }
  if (e->path == PATH_WALK4 && !e->keep && !(getenv("BPPGPU_WALK4C") && atoi(getenv("BPPGPU_WALK4C")) == 0)) {
    // walk4c: the same walk with leaf pushes in the register slot, tables cut into fixed-size chunks in walk order, the
    // program (descriptor words + chunk records) in the kernel-parameter block
    const int W = e->ncodes * e->ncodes;
    const int blk_int = C * 128, blk_tip = C * e->ncodes * 32, blk_wide = w4c_wide_block_bytes(C, W);
    // chunk geometry: bytes of tables and tip-code rows per ring stage (tuning knobs; a stage must hold the largest op)
    int CH = getenv("BPPGPU_WALK4_CH") ? std::max(1024, atoi(getenv("BPPGPU_WALK4_CH")) & ~127) : 8192;
    // Folded cherries: a cherry whose father is binary becomes a wide tip of the father (walk4c_kernels.cuh), its op leaves
    // the walk.  W <= 64 code pairs keep a row code in one byte and a wide block (C W 36 bytes) small next to the chunk; a
    // father whose op would outgrow the chunk keeps its second cherry as it is.  The fathers stay binary, so every op with a
    // wide tip is one of the binary shapes.  BPPGPU_W4C_FRONTIER=0 folds none (the program of the unfolded walk).
    e->w4c_cherry.assign(nn, 0);
    if (W <= kW4cMaxWideCodes && !(getenv("BPPGPU_W4C_FRONTIER") && atoi(getenv("BPPGPU_W4C_FRONTIER")) == 0)) {
      auto sons = [&](int n) { return e->child_off[n + 1] - e->child_off[n]; };
      auto son = [&](int n, int j) { return e->children[e->child_off[n] + j]; };
      auto cherry = [&](int n) { return sons(n) == 2 && e->leaf_slot[son(n, 0)] >= 0 && e->leaf_slot[son(n, 1)] >= 0; };
      for (int f = 0; f < nn; ++f) {
        if (sons(f) != 2) continue;
        for (int j = 0; j < 2; ++j) e->w4c_cherry[son(f, j)] = cherry(son(f, j));
        for (int j = 1; j >= 0; --j) {
          int b = 0;
          for (int k = 0; k < 2; ++k) {
            const int ch = son(f, k);
            b += e->w4c_cherry[ch] ? blk_wide : e->leaf_slot[ch] >= 0 ? blk_tip : blk_int;
          }
          if (b > CH) e->w4c_cherry[son(f, j)] = 0;
        }
      }
    }
    build_program(e, e->prog4c, false, true, &e->w4c_cherry);
    auto child_bytes = [&](const Child& ch) { return ch.kind != CHILD_TIP ? blk_int : ch.idx >= 0 ? blk_tip : blk_wide; };
    int max_op = 0, max_tips_op = 0;
    bool ok = e->prog4c.nslots <= 63;
    for (const Op& op : e->prog4c.ops) {
      int b = 0, nt = 0;
      for (int j = 0; j < op.nchild; ++j) {
        const Child& ch = e->prog4c.childs[op.child_begin + j];
        b += child_bytes(ch);
        nt += ch.kind == CHILD_TIP;
      }
      max_op = std::max(max_op, b);
      max_tips_op = std::max(max_tips_op, nt);
      if (op.nchild > 6) ok = false;
    }
    while (CH < max_op) CH *= 2;
    e->w4c_max_tips = getenv("BPPGPU_WALK4_MAXTIPS") ? std::max(1, std::min(31, atoi(getenv("BPPGPU_WALK4_MAXTIPS")))) : kW4cMaxTipsPerChunk;
    e->w4c_max_tips = std::max(e->w4c_max_tips, max_tips_op);
    if (e->w4c_max_tips > 31) ok = false;
    // launch plan.  Patterns per thread PT = 4 / 2 / 1 run 2 / 3 / 4 CTAs (of NW warps, 32 PT NW / C patterns) per SM; measured
    // on the 1024-taxon tree (ms per evaluation): 10.4 / 11.3 / 15.2 at 1M patterns, 1.47 / 1.56 / 1.98 at 125k -- PT = 4 wins at
    // every size that fills the GPU, so the default is ONE segment at the widest PT that has enough CTAs.  A launch is a
    // whole number of waves; BPPGPU_WALK4_PLAN=split walks k full waves at PT = 4 and the remainder with narrower CTAs
    // (measured on 125k patterns: 1.483 vs 1.469 ms -- the partial last wave of wide CTAs already runs at one CTA per SM and
    // is cheaper than a wave of narrow ones, so the split is not the default).  BPPGPU_WALK4_PT forces one segment.
    e->w4c_nw = C <= 4 ? 4 : 8;
    if (const char* env = getenv("BPPGPU_WALK4_NW")) {
      const int v = atoi(env);
      if ((v == 4 || v == 8) && v >= C) e->w4c_nw = v;
    }
    int forced_pt = 0;
    if (const char* env = getenv("BPPGPU_WALK4_PT")) {
      const int v = atoi(env);
      if (v >= 1 && v <= 4) forced_pt = v;
    }
    auto fits = [&](int pt) { return walk4c_smem_bytes(CH, e->prog4c.nslots, C, pt, e->w4c_nw, e->w4c_max_tips) <= 200 * 1024; };
    if (!fits(1)) ok = false;
    if (ok) {
      const int G = e->w4c_nw / C;
      auto ppc = [&](int pt) { return (long long)G * 32 * pt; };
      auto ctas_per_sm = [&](int pt) {
        const size_t smem = walk4c_smem_bytes(CH, e->prog4c.nslots, C, pt, e->w4c_nw, e->w4c_max_tips) + 1024;
        const int by_regs = e->w4c_nw == 8 ? (pt <= 2 ? 2 : 1) : (pt <= 1 ? 4 : pt <= 3 ? 3 : 2);   // walk4c_min_ctas + registers
        return std::max(1, std::min<int>(by_regs, (int)(227 * 1024 / smem)));
      };
      const double wave_ms[5] = {0, 0.287, 0.315, 0.36, 0.386};   // relative cost of one wave (only ratios matter)
      auto waves = [&](long long n, int pt) { const long long ctas = (n + ppc(pt) - 1) / ppc(pt); const long long slots = (long long)g_sm_count * ctas_per_sm(pt); return (ctas + slots - 1) / slots; };
      e->w4c_segs.clear();
      auto add_seg = [&](int pt, long long a, long long b) {
        if (b <= a) return;
        bppgpu_engine::W4cSeg sg{};
        sg.pt = pt; sg.pat0 = a; sg.pat_end = b;
        sg.grid = (int)((b - a + ppc(pt) - 1) / ppc(pt));
        e->w4c_segs.push_back(sg);
      };
      if (forced_pt) {
        int pt = forced_pt;
        while (pt > 1 && !fits(pt)) --pt;
        add_seg(pt, 0, N);
      } else if (N > 0 && !(getenv("BPPGPU_WALK4_PLAN") && !strncmp(getenv("BPPGPU_WALK4_PLAN"), "split", 5))) {
        int big = 4;
        while (big > 1 && (!fits(big) || N < (long long)g_sm_count * ctas_per_sm(big) * ppc(big))) big >>= 1;   // at least one wave
        add_seg(big, 0, N);
      } else if (N > 0) {
        int big = 4;
        while (big > 1 && !fits(big)) big >>= 1;
        const long long per_wave = (long long)g_sm_count * ctas_per_sm(big) * ppc(big);   // patterns in one full wave of the wide CTAs
        double best = 1e300;
        long long best_k = 0;
        int best_pt = 1;
        const long long kmax = N / per_wave;
        for (long long k = std::max<long long>(0, kmax - 1); k <= kmax; ++k)
          for (int pt : {1, 2, 4}) {
            if (pt > big || !fits(pt)) continue;
            const long long rem = N - k * per_wave;
            const double t = k * wave_ms[big] + (rem > 0 ? waves(rem, pt) * wave_ms[pt] : 0.0);
            if (t < best - 1e-12) { best = t; best_k = k; best_pt = pt; }
          }
        if (const char* pl = getenv("BPPGPU_WALK4_PLAN"))   // "split:<pt>[:<waves below the maximum>]" forces the remainder's PT (experiments)
          if (strlen(pl) > 6 && pl[5] == ':') {
            best_pt = std::max(1, std::min(big, atoi(pl + 6)));
            best_k = kmax;
            if (const char* c2 = strchr(pl + 6, ':')) best_k = std::max<long long>(0, kmax - atoi(c2 + 1));
          }
        if (best_pt == big && best_k == kmax) add_seg(big, 0, N);
        else { add_seg(big, 0, best_k * per_wave); add_seg(best_pt, best_k * per_wave, N); }
      }
      e->w4c_pt = e->w4c_segs.empty() ? 1 : e->w4c_segs[0].pt;
    }
    if (ok) {
      W4cProgram& W = e->w4c_prog;
      memset(&W, 0, sizeof(W));
      int nwords = 0, nchunks = 0, nops_in = 0, ntips_in = 0, tip0 = 0;
      size_t used = 0;
      auto close_chunk = [&]() {
        if (nchunks < kW4cMaxChunks) W.chunk[nchunks] = (unsigned)tip0 | ((unsigned)ntips_in << 16) | ((unsigned)nops_in << 21);
        ++nchunks;
        tip0 += ntips_in;
        nops_in = ntips_in = 0;
        used = 0;
      };
      for (const Op& op : e->prog4c.ops) {
        int b = 0, nt = 0;
        for (int j = 0; j < op.nchild; ++j) {
          const Child& ch = e->prog4c.childs[op.child_begin + j];
          b += child_bytes(ch);
          nt += ch.kind == CHILD_TIP;
        }
        if (nops_in == 31 || used + (size_t)b > (size_t)CH || ntips_in + nt > e->w4c_max_tips) close_chunk();
        auto kind4c = [](int k) { return k == CHILD_TIP ? W4C_TIP : k == CHILD_SLOT ? W4C_SLOT : k == CHILD_RSLOT ? W4C_RSL : W4C_REG; };
        int shape = W4C_GENERIC;
        int order[8] = {0, 1, 2, 3, 4, 5, 6, 7};   // order in which the handler consumes the children's table blocks
        unsigned jslot = 0, wide = 0;
        if (op.nchild == 2) {
          const Child& ca = e->prog4c.childs[op.child_begin];
          const Child& cb2 = e->prog4c.childs[op.child_begin + 1];
          const int ka = kind4c(ca.kind), kb = kind4c(cb2.kind);
          const bool wa = ka == W4C_TIP && ca.idx < 0, wb = kb == W4C_TIP && cb2.idx < 0;
          // a wide tip is consumed first (W4C_WA); two wide tips set both bits
          if (ka == W4C_TIP && kb == W4C_TIP) {
            shape = W4C_TT;
            if (wb && !wa) { order[0] = 1; order[1] = 0; }
            wide = (wa || wb ? (unsigned)W4C_WA : 0u) | (wa && wb ? (unsigned)W4C_WB : 0u);
          }
          else if (ka == W4C_TIP && kb == W4C_REG) { shape = W4C_TS; wide = wa ? (unsigned)W4C_WA : 0u; }
          else if (ka == W4C_REG && kb == W4C_TIP) { shape = W4C_TS; order[0] = 1; order[1] = 0; wide = wb ? (unsigned)W4C_WA : 0u; }
          else if (ka == W4C_RSL && kb == W4C_REG) shape = W4C_JW;
          else if (ka == W4C_REG && kb == W4C_RSL) { shape = W4C_JW; order[0] = 1; order[1] = 0; }
          else if (ka == W4C_SLOT && kb == W4C_REG) { shape = W4C_JS; jslot = (unsigned)ca.idx; }
          else if (ka == W4C_REG && kb == W4C_SLOT) { shape = W4C_JS; jslot = (unsigned)cb2.idx; order[0] = 1; order[1] = 0; }
        }
        unsigned d = (unsigned)shape | wide | (op.dst_slot == -2 ? (unsigned)W4C_DSTW : 0u) | ((unsigned)op.nchild << 24);
        if (op.dst_slot >= 0) d |= ((unsigned)op.dst_slot << 8) | 0x4000u;
        unsigned d2 = 0;
        int nslot_tok = 0;
        if (shape != W4C_GENERIC) d |= jslot << 16;
        for (int jj = 0; jj < op.nchild; ++jj) {
          const int j = order[jj];
          const Child& ch = e->prog4c.childs[op.child_begin + j];
          if (shape == W4C_GENERIC) {
            d2 |= (unsigned)kind4c(ch.kind) << (2 * j);
            if (ch.kind == CHILD_SLOT) d2 |= (unsigned)ch.idx << (12 + 6 * nslot_tok++);
          }
          if (shape == W4C_GENERIC && ch.kind == CHILD_TIP && ch.idx < 0) ok = false;   // (the fathers of cherries are binary)
          Pack4cBlock pb{};
          pb.kind = kind4c(ch.kind);
          pb.pnode = ch.pnode;
          pb.son0 = pb.son1 = -1;
          pb.off = (long long)((size_t)nchunks * CH + used);
          if (ch.kind == CHILD_TIP && ch.idx < 0) {
            pb.kind = W4C_CHERRY;
            pb.son0 = e->children[e->child_off[ch.pnode]];
            pb.son1 = e->children[e->child_off[ch.pnode] + 1];
            e->w4c_tip_order.push_back(make_int2(e->leaf_slot[pb.son0], e->leaf_slot[pb.son1]));
          } else if (ch.kind == CHILD_TIP) {
            e->w4c_tip_order.push_back(make_int2(ch.idx, -1));
          }
          e->w4c_blocks.push_back(pb);
          used += (size_t)child_bytes(ch);
        }
        if (nslot_tok > 3) ok = false;
        if (nwords < kW4cMaxOps) W.desc[nwords] = make_uint2(d, d2);
        ++nwords;
        ++nops_in;
        ntips_in += nt;
      }
      close_chunk();
      if (nwords > kW4cMaxOps || nchunks > kW4cMaxChunks || e->w4c_tip_order.size() > 65535) ok = false;
      e->w4c_nchunks = nchunks;
      e->w4c_CH = CH;
      e->w4c_stream_bytes = (size_t)nchunks * CH;
      e->w4c = ok;
      e->w4c_frontier_nodes = ok ? (int)std::count(e->w4c_cherry.begin(), e->w4c_cherry.end(), 1) : 0;
    }
  }
  int rc = upload_program(e, e->prog);
  if (rc) return rc;
  rc = upload_program(e, e->gprog);
  if (rc) return rc;
  // siblings per node (generic kinds) for the prefix pass
  e->sib_off.assign(nn + 1, 0);
  std::vector<Child> allsibs;
  for (int n = 0; n < nn; ++n) {
    e->sib_off[n] = (int)allsibs.size();
    if (n == e->root) continue;
    int f = e->parent[n];
    for (int k = e->child_off[f]; k < e->child_off[f + 1]; ++k) {
      int b = e->children[k];
      if (b == n) continue;
      Child c{};
      c.pnode = b;
      if (e->leaf_slot[b] >= 0) { c.kind = CHILD_TIP; c.idx = e->leaf_slot[b]; }
      else { c.kind = CHILD_KEEP; c.idx = e->internal_idx[b]; }
      allsibs.push_back(c);
    }
  }
  e->sib_off[nn] = (int)allsibs.size();
  e->sibs_flat = allsibs;
  BPP_CUDA(dev_alloc(e, &e->d_sibs, allsibs.size()));
  if (!allsibs.empty())
    BPP_CUDA(cudaMemcpy(e->d_sibs, allsibs.data(), allsibs.size() * sizeof(Child), cudaMemcpyHostToDevice));

  // ---- buffers ------------------------------------------------------------------------
  const size_t SS = (size_t)S * S;
  BPP_CUDA(dev_alloc(e, (unsigned char**)&e->d_codes, (size_t)e->nl * N * e->code_bytes));
  BPP_CUDA(cudaMemset(e->d_codes, 0, std::max<size_t>(1, (size_t)e->nl * N * e->code_bytes)));
  BPP_CUDA(dev_alloc(e, &e->d_code_table, (size_t)e->ncodes * S));
  BPP_CUDA(cudaMemcpy(e->d_code_table, cfg->code_table, (size_t)e->ncodes * S * 8, cudaMemcpyHostToDevice));
  {
    std::vector<int> single(e->ncodes, -1);
    for (int k = 0; k < e->ncodes; ++k) {
      int ones = 0, other = 0, pos = -1;
      for (int x = 0; x < S; ++x) {
        const double v = cfg->code_table[(size_t)k * S + x];
        if (v == 1.0) { ++ones; pos = x; }
        else if (v != 0.0) ++other;
      }
      if (ones == 1 && other == 0) single[k] = pos;
    }
    BPP_CUDA(dev_alloc(e, &e->d_code_single, (size_t)e->ncodes));
    BPP_CUDA(cudaMemcpy(e->d_code_single, single.data(), e->ncodes * sizeof(int), cudaMemcpyHostToDevice));
    e->h_code_single = single;
    e->h_code_table.assign(cfg->code_table, cfg->code_table + (size_t)e->ncodes * S);
  }
  BPP_CUDA(dev_alloc(e, &e->d_weights, (size_t)N));
  BPP_CUDA(dev_alloc(e, &e->d_rates, (size_t)C));
  BPP_CUDA(dev_alloc(e, &e->d_probs, (size_t)C));
  BPP_CUDA(dev_alloc(e, &e->d_rootfreq, (size_t)e->npoints * S));
  BPP_CUDA(dev_alloc(e, &e->d_rootfreq_used, (size_t)e->npoints * S));
  BPP_CUDA(dev_alloc(e, &e->d_brlen, (size_t)e->npoints * nn));
  BPP_CUDA(cudaMemset(e->d_brlen, 0, (size_t)e->npoints * nn * 8));
  BPP_CUDA(dev_alloc(e, &e->d_branch_model, (size_t)e->npoints * nn));
  BPP_CUDA(dev_alloc(e, &e->d_leaf_nodes, (size_t)e->nl));
  BPP_CUDA(cudaMemcpy(e->d_leaf_nodes, e->leaf_nodes.data(), e->nl * sizeof(int), cudaMemcpyHostToDevice));
  e->models.resize(e->nmodels);
  BPP_CUDA(dev_alloc(e, &e->d_models, (size_t)e->nmodels));
  e->h_brlen.assign((size_t)e->npoints * nn, 0.0);
  e->h_branch_model.assign((size_t)e->npoints * nn, 0);
  if (e->nmodels == e->npoints && e->npoints > 1)
    for (int p = 0; p < e->npoints; ++p)
      for (int n = 0; n < nn; ++n) e->h_branch_model[(size_t)p * nn + n] = p;
  BPP_CUDA(cudaMemcpy(e->d_branch_model, e->h_branch_model.data(), e->h_branch_model.size() * sizeof(int),
                      cudaMemcpyHostToDevice));
  e->have_tip.assign(e->nl, 0);
  e->have_brlen.assign(e->npoints, 0);
  e->have_rootfreq.assign(e->npoints, 0);

  // P tables: as many points per chunk as fit a 16 GiB budget
  const size_t per_point = (size_t)nn * C * SS * 8;
  size_t budget = (size_t)16 << 30;
  if (e->path == PATH_POINTS) {
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) == cudaSuccess) budget = std::max(budget, fr / 2);
  }
  // one character, one class, many points: the factored route needs no tables (they are allocated on demand, for the points
  // the guard sends to the table route); KEEP_CLVS asks for the per-node arrays, which only the table route has
  e->chr_factored = e->path == PATH_POINTS && N == 1 && C == 1 && S <= 8 * kChrWarps * kChrMaxRB && !(cfg->flags & BPPGPU_FLAG_KEEP_CLVS) &&
                    !(getenv("BPPGPU_POINTS_FACTORED") && atoi(getenv("BPPGPU_POINTS_FACTORED")) == 0);
  if (e->chr_factored) {
    e->tables_allocated = false;
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) fr = (size_t)8 << 30;
    const size_t per_pt = (size_t)nn * S * 8 + (size_t)nn * 4;
    e->fchunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)e->npoints, (fr / 4) / per_pt));
    BPP_CUDA(dev_alloc(e, &e->d_chr_term, (size_t)e->fchunk * nn * S));
    BPP_CUDA(dev_alloc(e, &e->d_chr_term_exp, (size_t)e->fchunk * nn));
    e->gchunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)e->npoints, ((size_t)1 << 30) / (3 * SS * 8)));
    BPP_CUDA(dev_alloc(e, &e->d_chr_guardP, (size_t)e->gchunk * 3 * SS));
    BPP_CUDA(dev_alloc(e, &e->d_chr_bad, (size_t)e->npoints));
    BPP_CUDA(dev_alloc(e, &e->d_chr_probe_t, (size_t)e->npoints * 3));
    BPP_CUDA(dev_alloc(e, &e->d_chr_probe_bm, (size_t)e->npoints * 3));
    BPP_CUDA(dev_alloc(e, &e->d_models_noclamp, (size_t)e->nmodels));
    BPP_CUDA(dev_alloc(e, &e->d_chr_leaf_state, (size_t)nn));
    BPP_CUDA(dev_alloc(e, &e->d_chr_leaf_vec, (size_t)nn * S));
    BPP_CUDA(dev_alloc(e, &e->d_child_off, (size_t)nn + 1));
    BPP_CUDA(dev_alloc(e, &e->d_children, e->children.size()));
    BPP_CUDA(cudaMemcpy(e->d_child_off, e->child_off.data(), (nn + 1) * sizeof(int), cudaMemcpyHostToDevice));
    if (!e->children.empty()) BPP_CUDA(cudaMemcpy(e->d_children, e->children.data(), e->children.size() * sizeof(int), cudaMemcpyHostToDevice));
    const int maxtiles = nn;   // generous: a tile holds at least one edge
    BPP_CUDA(dev_alloc(e, &e->d_chr_tile_edges, (size_t)maxtiles * kChrCols));
    BPP_CUDA(dev_alloc(e, &e->d_chr_tile_kind, (size_t)maxtiles));
    e->h_codes.assign(e->nl, 0);
    BPP_CUDA(cudaFuncSetAttribute(chr_level_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)chr_level_smem(S)));
    BPP_CUDA(cudaFuncSetAttribute(chr_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)std::max(chr_level_smem(S), (size_t)116 * 1024)));
    {
      const bool slab_on = !(getenv("BPPGPU_CHR_SLAB") && atoi(getenv("BPPGPU_CHR_SLAB")) == 0);   // read per engine (A/B tests)
      const int K8 = (S + 7) & ~7;
      e->chr_slab = slab_on && K8 <= 8 * kChrCons * kChrMaxRB;
      if (e->chr_slab) {
        BPP_CUDA(dev_alloc(e, &e->d_chr_aslab, (size_t)e->nmodels * 3 * K8 * K8));   // [V^-1 | V] slab images + (V^-1)^T
        const int optin = (int)std::min<size_t>((size_t)g_smem_optin, chr_slab_smem(S, kChrMaxStages));
        BPP_CUDA(cudaFuncSetAttribute(chr_level_slab_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
        BPP_CUDA(cudaFuncSetAttribute(chr_chain_slab_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
        BPP_CUDA(cudaFuncSetAttribute(chr_chain_slab_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
      }
    }
    e->pchunk = 1;
  } else {
    e->pchunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)e->npoints, budget / std::max<size_t>(1, (e->path == PATH_POINTS ? 1 : 3) * per_point)));
    BPP_CUDA(dev_alloc(e, &e->d_P, (size_t)e->pchunk * nn * C * SS));
  }
  if (e->path == PATH_WALK4 && !e->w4c) {
    BPP_CUDA(dev_alloc(e, &e->d_w4_desc, e->w4_desc.size()));
    BPP_CUDA(cudaMemcpy(e->d_w4_desc, e->w4_desc.data(), e->w4_desc.size() * 8, cudaMemcpyHostToDevice));
    BPP_CUDA(dev_alloc(e, &e->d_w4_tip_order, e->w4_tip_order.size()));
    BPP_CUDA(cudaMemcpy(e->d_w4_tip_order, e->w4_tip_order.data(), e->w4_tip_order.size() * 4, cudaMemcpyHostToDevice));
    BPP_CUDA(dev_alloc(e, &e->d_w4_blocks, e->w4_blocks.size()));
    BPP_CUDA(cudaMemcpy(e->d_w4_blocks, e->w4_blocks.data(), e->w4_blocks.size() * sizeof(PackBlock), cudaMemcpyHostToDevice));
    BPP_CUDA(dev_alloc(e, &e->d_w4_stream, (size_t)e->pchunk * e->w4_stream_len + (size_t)e->ncodes * C * 4 + 64 + 8192));
    BPP_CUDA(cudaMemset(e->d_w4_stream, 0, ((size_t)e->pchunk * e->w4_stream_len + (size_t)e->ncodes * C * 4 + 64 + 8192) * 8));
    BPP_CUDA(dev_alloc(e, &e->d_codesT, (size_t)N * e->w4_tstride));
  }
  if (e->w4c) {
    BPP_CUDA(dev_alloc(e, &e->d_w4c_stream, (size_t)e->pchunk * e->w4c_stream_bytes));
    BPP_CUDA(cudaMemset(e->d_w4c_stream, 0, (size_t)e->pchunk * e->w4c_stream_bytes));
    BPP_CUDA(dev_alloc(e, &e->d_w4c_blocks, e->w4c_blocks.size()));
    BPP_CUDA(cudaMemcpy(e->d_w4c_blocks, e->w4c_blocks.data(), e->w4c_blocks.size() * sizeof(Pack4cBlock), cudaMemcpyHostToDevice));
    BPP_CUDA(dev_alloc(e, &e->d_w4c_tip_order, e->w4c_tip_order.size()));
    BPP_CUDA(cudaMemcpy(e->d_w4c_tip_order, e->w4c_tip_order.data(), e->w4c_tip_order.size() * sizeof(int2), cudaMemcpyHostToDevice));
    size_t codes_bytes = 0;
    int parts = 0;
    for (auto& sg : e->w4c_segs) {
      sg.codes_off = codes_bytes;
      sg.part0 = parts;
      codes_bytes += (size_t)sg.grid * e->w4c_tip_order.size() * (size_t)(e->w4c_nw / C) * 32 * sg.pt;
      codes_bytes = (codes_bytes + 127) & ~(size_t)127;
      parts += sg.grid;
    }
    BPP_CUDA(dev_alloc(e, &e->d_codesC, codes_bytes + 128));
    BPP_CUDA(dev_alloc(e, &e->d_w4c_counter, 1));
    BPP_CUDA(cudaMemset(e->d_w4c_counter, 0, sizeof(unsigned)));
  }
  if ((e->path != PATH_WALK4 || e->keep) && e->path != PATH_POINTS)
    BPP_CUDA(dev_alloc(e, &e->d_tiptab, (size_t)e->pchunk * e->nl * C * e->ncodes * S));

  const size_t clv = (size_t)N * C * S;
  if (e->keep && e->tables_allocated) {
    const size_t mult = e->path == PATH_POINTS ? (size_t)e->pchunk : 1;
    BPP_CUDA(dev_alloc(e, &e->d_keep, mult * e->ni * clv));
    BPP_CUDA(dev_alloc(e, &e->d_keep_exp, mult * e->ni * N * C));
  }
  if (e->path == PATH_WALKS && e->prog.nslots > 0) {
    BPP_CUDA(dev_alloc(e, &e->d_gstack, (size_t)e->prog.nslots * clv));
    BPP_CUDA(dev_alloc(e, &e->d_gstack_exp, (size_t)e->prog.nslots * N * C));
  }
  BPP_CUDA(dev_alloc(e, &e->d_SR, (size_t)N));
  BPP_CUDA(dev_alloc(e, &e->d_rexp, (size_t)N));
  BPP_CUDA(dev_alloc(e, &e->d_site_lnl, (size_t)e->npoints * N));
  const long long rows = N * C;
  e->n_partials = (int)std::max<long long>(1, std::max((rows + 127) / 128, (N + 255) / 256) + 1);
  BPP_CUDA(dev_alloc(e, &e->d_partials, (size_t)e->n_partials));
  BPP_CUDA(dev_alloc(e, &e->d_partials2, (size_t)e->n_partials));
  BPP_CUDA(dev_alloc(e, &e->d_out, (size_t)e->npoints * (1 + 2 * nn)));
  BPP_CUDA(cudaMemset(e->d_out, 0, (size_t)e->npoints * (1 + 2 * nn) * 8));
  BPP_CUDA(dev_alloc(e, &e->d_status, 1));
  BPP_CUDA(cudaMemset(e->d_status, 0, sizeof(int)));
  BPP_CUDA(dev_alloc(e, &e->d_wr_recs, (size_t)S + 1));
  BPP_CUDA(cudaEventCreateWithFlags(&e->eval_done, cudaEventDisableTiming));

  // S = 20 on the FP64 tensor cores: fragment-order operands, one persistent CTA per SM (dmma_family_kernels.cuh);
  // BPPGPU_FAMILY=0 keeps the older per-node / per-branch kernels
  {
    const char* fenv = getenv("BPPGPU_FAMILY");
    e->family = e->path == PATH_DMMA && S == 20 && C <= kFamMaxClasses && N > 0 && e->npoints == 1 && !(fenv && atoi(fenv) == 0);
  }
  if (e->family) {
    // The S = 20 kernels own their CLV slabs, so when no node needs the first-generation kernels (every father has <= 3
    // sons) the slabs are CLASS-MAJOR [class][pattern][state]: the 8 rows of an item are then 1280 contiguous bytes instead
    // of 160-byte pieces at a 160 C stride.  Accessors transpose back to the reference's [pattern][class][state].
    bool wide = false;
    for (int n = 0; n < nn; ++n)
      if (e->child_off[n + 1] - e->child_off[n] > kFamMaxSons) wide = true;
    const char* lenv = getenv("BPPGPU_CLV_LAYOUT");  // "pattern" keeps the reference order (A/B measurements)
    e->clv_class_major = !wide && !wroot && (double)N * C * S < 2.0e9 && !(lenv && !strcmp(lenv, "pattern"));
    if ((double)N * C * S >= 2.0e9) e->family = false;  // 32-bit row offsets inside the kernels
  }
  {
    // S = 64 (codon), one rate class: the same fragment-order pruning kernel (the derivative pass keeps the first-generation
    // kernels, which share the reference-order slabs: with C = 1 both orders coincide)
    const char* fenv = getenv("BPPGPU_FAMILY");
    e->prune64 = e->path == PATH_DMMA && S == 64 && C == 1 && N > 0 && e->npoints == 1 && (double)N * C * S < 2.0e9 &&
                 !(fenv && atoi(fenv) == 0);
  }
  if (e->family || e->prune64) {
    long long slots = g_sm_count;
    if (const char* env = getenv("BPPGPU_FAMILY_GRID")) slots = std::max(1, atoi(env));  // test knob: few CTAs, long ranges
    long long ppc = (N + slots - 1) / slots;
    ppc = std::max<long long>(8, (ppc + 7) / 8 * 8);
    e->fam_ppc = (int)ppc;
    e->fam_grid = (int)((N + ppc - 1) / ppc);
    BPP_CUDA(dev_alloc(e, &e->d_fam_packL, (size_t)nn * C * prune_pack(S)));
    auto attr = [](auto k, size_t smem) { return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); };
    if (e->family) {
      if (const char* env = getenv("BPPGPU_PRUNE_CFG")) e->prune_cfg = std::min(2, std::max(0, atoi(env)));
#define BPP_PRUNE_ATTR(Kv) \
      BPP_CUDA(attr(dmma_prune_kernel<20, Kv, 0>, dmma_prune_smem<20, Kv, 0>(C))); \
      BPP_CUDA(attr(dmma_prune_level_kernel<20, Kv, 0>, dmma_prune_smem<20, Kv, 0>(C))); \
      BPP_CUDA(attr(dmma_prune_kernel<20, Kv, 1>, dmma_prune_smem<20, Kv, 1>(C))); \
      BPP_CUDA(attr(dmma_prune_kernel<20, Kv, 2>, dmma_prune_smem<20, Kv, 2>(C)));
      BPP_PRUNE_ATTR(0) BPP_PRUNE_ATTR(1) BPP_PRUNE_ATTR(2) BPP_PRUNE_ATTR(3)
#undef BPP_PRUNE_ATTR
      BPP_CUDA(attr(dmma_prune_kernel<20, 4, 0>, dmma_prune_smem<20, 4, 0>(C)));
      BPP_CUDA(attr(dmma_prune_level_kernel<20, 4, 0>, dmma_prune_smem<20, 4, 0>(C)));
    } else {
      BPP_CUDA(attr(dmma_prune_kernel<64, 0, 0>, dmma_prune_smem<64, 0, 0>(C)));
      BPP_CUDA(attr(dmma_prune_kernel<64, 1, 0>, dmma_prune_smem<64, 1, 0>(C)));
      BPP_CUDA(attr(dmma_prune_kernel<64, 2, 0>, dmma_prune_smem<64, 2, 0>(C)));
      BPP_CUDA(attr(dmma_prune_kernel<64, 3, 0>, dmma_prune_smem<64, 3, 0>(C)));
      BPP_CUDA(attr(dmma_prune_kernel<64, 4, 0>, dmma_prune_smem<64, 4, 0>(C)));
      BPP_CUDA(attr(dmma_prune_level_kernel<64, 0, 0>, dmma_prune_smem<64, 0, 0>(C)));
      BPP_CUDA(attr(dmma_prune_level_kernel<64, 1, 0>, dmma_prune_smem<64, 1, 0>(C)));
      BPP_CUDA(attr(dmma_prune_level_kernel<64, 2, 0>, dmma_prune_smem<64, 2, 0>(C)));
      BPP_CUDA(attr(dmma_prune_level_kernel<64, 3, 0>, dmma_prune_smem<64, 3, 0>(C)));
      BPP_CUDA(attr(dmma_prune_level_kernel<64, 4, 0>, dmma_prune_smem<64, 4, 0>(C)));
    }
    {
      // level-batched pruning launches (dmma_prune_level_kernel): one point, every node within the kernels' son limit
      const bool lb_on = !(getenv("BPPGPU_LEVEL_BATCH") && atoi(getenv("BPPGPU_LEVEL_BATCH")) == 0);   // read per engine (A/B tests)
      e->level_batch = lb_on && e->npoints == 1 && e->prune_cfg == 0;
      for (const Op& op : e->gprog.ops)
        if (op.nchild > kFamMaxSons) e->level_batch = false;
      if (e->level_batch) BPP_CUDA(dev_alloc(e, &e->d_prune_nodes, e->gprog.ops.size()));
      if (e->level_batch && e->family) BPP_CUDA(dev_alloc(e, &e->d_family_nodes, (size_t)e->nn));
    }
  }

  if (e->w4c) {
    for (int pt = 1; pt <= 4; ++pt) {   // opt in to the dynamic shared memory of every instantiation a plan may use
      const size_t smem = walk4c_smem_bytes(e->w4c_CH, e->prog4c.nslots, C, pt, e->w4c_nw, e->w4c_max_tips);
      if (smem > 200 * 1024) continue;
      int rc4 = walk4c_dispatch(e, pt, nullptr, 0, smem, nullptr, true);
      if (rc4) return rc4;
    }
    e->stats.stack_slots = e->prog4c.nslots;
  } else if (e->path == PATH_WALK4) {
    // patterns per thread: 2 (4 CTAs of 128 threads per SM at 128 registers) while the stack leaves room for it
    e->w4_pt = 2;
    while (e->w4_pt > 1 && (size_t)e->prog.nslots * e->w4_pt * kWalk4Threads * 36 > 56 * 1024) e->w4_pt >>= 1;
    if (N * C < (long long)g_sm_count * 4 * kWalk4Threads * 4) e->w4_pt = 1;  // small inputs: more CTAs instead
    if (const char* env = getenv("BPPGPU_WALK4_PT")) {  // tuning knob: 1, 2 or 4
      const int v = atoi(env);
      if (v >= 1 && v <= 4 && (size_t)e->prog.nslots * v * kWalk4Threads * 36 <= 200 * 1024) e->w4_pt = v;
    }
    int rc4 = walk4_dispatch(e, nullptr, 0, 0, nullptr, true);
    if (rc4) return rc4;
  }
  if (e->path == PATH_WALKS) {
    size_t smem = (size_t)kMaxStagedChildren * C * (S * S + 2) * 8;
    switch (ilog2(C)) {
      case 0: BPP_CUDA(cudaFuncSetAttribute(walkS_kernel<20, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
      case 1: BPP_CUDA(cudaFuncSetAttribute(walkS_kernel<20, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
      case 2: BPP_CUDA(cudaFuncSetAttribute(walkS_kernel<20, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
      default: BPP_CUDA(cudaFuncSetAttribute(walkS_kernel<20, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); break;
    }
  }
  e->stats.path = e->path;
  if (!e->w4c) e->stats.stack_slots = e->prog.nslots;
  e->stats.hbm_bytes_resident = (int64_t)e->bytes_resident;
  return BPPGPU_OK;
}

int bppgpu_create(const bppgpu_config* cfg, bppgpu_engine** out) {
  if (!cfg || !out) BPP_FAIL(BPPGPU_E_INVALID, "null argument");
  *out = nullptr;
  if (cfg->n_states <= 0 || cfg->n_cats <= 0 || cfg->n_patterns < 0 || cfg->n_nodes <= 1 || cfg->n_points <= 0 ||
      cfg->n_models <= 0 || cfg->n_codes <= 0)
    BPP_FAIL(BPPGPU_E_INVALID, "non-positive dimension in bppgpu_config");
  if (cfg->root < 0 || cfg->root >= cfg->n_nodes) BPP_FAIL(BPPGPU_E_INVALID, "root id out of range");
  if (cfg->code_bytes != 1 && cfg->code_bytes != 2) BPP_FAIL(BPPGPU_E_INVALID, "code_bytes must be 1 or 2");
  if (cfg->code_bytes == 1 && cfg->n_codes > 256) BPP_FAIL(BPPGPU_E_INVALID, "n_codes > 256 needs code_bytes = 2");
  if (!cfg->child_offsets || !cfg->children || !cfg->code_table) BPP_FAIL(BPPGPU_E_INVALID, "null array in bppgpu_config");
  int rc = check_device(cfg->device);
  if (rc) return rc;
  bppgpu_engine* e = new bppgpu_engine();
  rc = create_impl(cfg, e);
  if (rc) {
    std::string msg = last_error();
    bppgpu_destroy(e);
    last_error() = msg;
    return rc;
  }
  *out = e;
  return BPPGPU_OK;
}

#define ENGINE_ENTER(e)                                                \
  if (!(e)) BPP_FAIL(BPPGPU_E_INVALID, "null engine");                 \
  BPP_CUDA(cudaSetDevice((e)->dev));
// setters and accessors: additionally wait for the last evaluation, whatever stream it was enqueued on (bppgpu_eval_device
// does not synchronise), before engine buffers are read or overwritten
#define ENGINE_SYNC(e)                                                 \
  ENGINE_ENTER(e);                                                     \
  if ((e)->eval_done) BPP_CUDA(cudaEventSynchronize((e)->eval_done));

// tip codes index the per-branch tip tables directly: reject anything outside [0, n_codes) at upload, naming leaf and pattern
static int check_codes(bppgpu_engine* e, const void* codes, long long n, int leaf_node_or_minus1) {
  long long bad = -1;
  if (e->code_bytes == 1) {
    if (e->ncodes < 256) {
      const unsigned char* c = (const unsigned char*)codes;
      for (long long i = 0; i < n; ++i)
        if (c[i] >= e->ncodes) { bad = i; break; }
    }
  } else {
    const unsigned short* c = (const unsigned short*)codes;
    for (long long i = 0; i < n; ++i)
      if (c[i] >= e->ncodes) { bad = i; break; }
  }
  if (bad < 0) return BPPGPU_OK;
  const int leaf = leaf_node_or_minus1 >= 0 ? leaf_node_or_minus1 : e->leaf_nodes[(size_t)(bad / std::max<long long>(1, e->N))];
  BPP_FAIL(BPPGPU_E_INVALID, "tip code out of range at leaf node %d, pattern %lld: the code table has %d rows", leaf,
           bad % std::max<long long>(1, e->N), e->ncodes);
}

int bppgpu_set_tip_codes(bppgpu_engine* e, int32_t node, const void* codes) {
  ENGINE_SYNC(e);
  if (node < 0 || node >= e->nn || e->leaf_slot[node] < 0) BPP_FAIL(BPPGPU_E_INVALID, "node %d is not a leaf", node);
  if (!codes) BPP_FAIL(BPPGPU_E_INVALID, "null codes");
  if (int rc = check_codes(e, codes, e->N, node)) return rc;
  const size_t bytes = (size_t)e->N * e->code_bytes;
  BPP_CUDA(cudaMemcpyAsync((unsigned char*)e->d_codes + (size_t)e->leaf_slot[node] * bytes, codes, bytes,
                           cudaMemcpyHostToDevice, e->stream));
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  e->have_tip[e->leaf_slot[node]] = 1;
  if (e->chr_factored) {
    e->h_codes[(size_t)e->leaf_slot[node]] = e->code_bytes == 1 ? *(const unsigned char*)codes : *(const unsigned short*)codes;
    e->chr_tiles_dirty = true;
  }
  e->codesT_dirty = true;
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_set_all_tip_codes(bppgpu_engine* e, const void* codes) {
  ENGINE_SYNC(e);
  if (!codes) BPP_FAIL(BPPGPU_E_INVALID, "null codes");
  if (int rc = check_codes(e, codes, e->N * e->nl, -1)) return rc;
  const size_t bytes = (size_t)e->N * e->code_bytes * e->nl;
  BPP_CUDA(cudaMemcpyAsync(e->d_codes, codes, bytes, cudaMemcpyHostToDevice, e->stream));
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  std::fill(e->have_tip.begin(), e->have_tip.end(), 1);
  if (e->chr_factored) {
    for (int l = 0; l < e->nl; ++l)
      e->h_codes[(size_t)l] = e->code_bytes == 1 ? ((const unsigned char*)codes)[l] : ((const unsigned short*)codes)[l];
    e->chr_tiles_dirty = true;
  }
  e->codesT_dirty = true;
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_leaf_slot(bppgpu_engine* e, int32_t node, int32_t* slot) {
  if (!e || !slot) BPP_FAIL(BPPGPU_E_INVALID, "null argument");
  if (node < 0 || node >= e->nn) BPP_FAIL(BPPGPU_E_INVALID, "node out of range");
  *slot = e->leaf_slot[node];
  return BPPGPU_OK;
}

int bppgpu_set_pattern_weights(bppgpu_engine* e, const uint32_t* w) {
  ENGINE_SYNC(e);
  if (!w && e->N > 0) BPP_FAIL(BPPGPU_E_INVALID, "null weights");
  std::vector<double> wd((size_t)e->N);
  for (long long i = 0; i < e->N; ++i) wd[i] = (double)w[i];
  BPP_CUDA(cudaMemcpy(e->d_weights, wd.data(), (size_t)e->N * 8, cudaMemcpyHostToDevice));
  e->have_weights = true;
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_set_rates(bppgpu_engine* e, const double* rates, const double* probs) {
  ENGINE_SYNC(e);
  if (!rates || !probs) BPP_FAIL(BPPGPU_E_INVALID, "null rates / probs");
  e->h_rates.assign(rates, rates + e->C);
  e->h_probs.assign(probs, probs + e->C);
  BPP_CUDA(cudaMemcpy(e->d_rates, rates, e->C * 8, cudaMemcpyHostToDevice));
  BPP_CUDA(cudaMemcpy(e->d_probs, probs, e->C * 8, cudaMemcpyHostToDevice));
  e->have_rates = true;
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_set_model(bppgpu_engine* e, int32_t slot, const bppgpu_model_desc* m) {
  ENGINE_SYNC(e);
  if (!m) BPP_FAIL(BPPGPU_E_INVALID, "null model");
  if (slot < 0 || slot >= e->nmodels) BPP_FAIL(BPPGPU_E_INVALID, "model slot %d out of range", slot);
  if (m->n_states != e->S) BPP_FAIL(BPPGPU_E_INVALID, "model has %d states, engine %d", m->n_states, e->S);
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  int rc = upload_model(e->models[slot], m, e->S, e->path != PATH_POINTS);
  if (rc) return rc;
  e->models_dirty = true;
  e->chr_slab_dirty = true;
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_set_models(bppgpu_engine* e, int32_t first_slot, int32_t n, const bppgpu_model_desc* descs) {
  ENGINE_SYNC(e);
  if (!descs || n < 0 || first_slot < 0 || first_slot + n > e->nmodels) BPP_FAIL(BPPGPU_E_INVALID, "bad slot range or null descriptors");
  const int S = e->S;
  for (int k = 0; k < n; ++k)
    if (descs[k].n_states != S) BPP_FAIL(BPPGPU_E_INVALID, "model %d has %d states, engine %d", k, descs[k].n_states, S);
  const size_t img_doubles = model_slab_doubles(S);
  // Several host threads, each with two pinned staging images and a stream of its own: model k is packed on the host while the
  // previous ones travel, and the packing itself (a few hundred KB of memcpy per model) is spread over the threads -- a batched-
  // points optimiser re-sends thousands of eigensystems per step (BASELINE config 5), and one thread packing 4096 x 640 KB was
  // most of that step's end-to-end time.
  constexpr int kMaxT = bppgpu_engine::kStageThreads;
  if (!e->h_stage) {
    BPP_CUDA(cudaMallocHost(&e->h_stage, (size_t)kMaxT * 2 * img_doubles * 8));
    for (int t = 0; t < kMaxT; ++t) {
      BPP_CUDA(cudaStreamCreateWithFlags(&e->stage_stream[t], cudaStreamNonBlocking));
      for (int b = 0; b < 2; ++b) BPP_CUDA(cudaEventCreateWithFlags(&e->stage_ev[t][b], cudaEventDisableTiming));
    }
  }
  static const int env_threads = getenv("BPPGPU_COPY_THREADS") ? atoi(getenv("BPPGPU_COPY_THREADS")) : (std::thread::hardware_concurrency() >= 16 ? 8 : 4);
  const int T = std::max(1, std::min({kMaxT, env_threads, n / 4 + 1, (int)std::max(1u, std::thread::hardware_concurrency())}));
  std::vector<int> rcs(T, BPPGPU_OK);
  std::vector<std::string> msgs(T);
  auto worker = [&](int t) -> int {
    BPP_CUDA(cudaSetDevice(e->dev));
    int it = 0;
    for (int k = t; k < n; k += T, ++it) {
      DevModel& dm = e->models[first_slot + k];
      const int b = it & 1;
      double* img = e->h_stage + ((size_t)t * 2 + b) * img_doubles;
      BPP_CUDA(cudaEventSynchronize(e->stage_ev[t][b]));   // the copy that last used this image has left
      size_t used = 0;
      bool padded = false;
      int rc = build_model_image(dm, &descs[k], S, e->path != PATH_POINTS, /*keep_q=*/e->path != PATH_POINTS, img, &used, &padded);
      if (rc) return rc;
      rc = ensure_model_storage(dm, S, padded);
      if (rc) return rc;
      rc = send_model_image(dm, S, img, used, padded, e->stage_stream[t]);
      if (rc) return rc;
      BPP_CUDA(cudaEventRecord(e->stage_ev[t][b], e->stage_stream[t]));
      dm.set = true;
    }
    BPP_CUDA(cudaStreamSynchronize(e->stage_stream[t]));
    return BPPGPU_OK;
  };
  auto run = [&](int t) {
    rcs[t] = worker(t);
    if (rcs[t]) msgs[t] = last_error();   // the error string is thread-local
  };
  std::vector<std::thread> th;
  for (int t = 1; t < T; ++t) th.emplace_back(run, t);
  run(0);
  for (auto& x : th) x.join();
  e->models_dirty = true;
  e->chr_slab_dirty = true;
  e->last_point = -1;
  for (int t = 0; t < T; ++t)
    if (rcs[t]) {
      for (int u = 0; u < T; ++u) cudaStreamSynchronize(e->stage_stream[u]);
      last_error() = msgs[t];
      return rcs[t];
    }
  return BPPGPU_OK;
}

int bppgpu_set_branch_models(bppgpu_engine* e, int32_t point, const int32_t* slot_of_node) {
  ENGINE_SYNC(e);
  if (point < 0 || point >= e->npoints || !slot_of_node) BPP_FAIL(BPPGPU_E_INVALID, "bad point or null array");
  for (int n = 0; n < e->nn; ++n) {
    if (n != e->root && (slot_of_node[n] < 0 || slot_of_node[n] >= e->nmodels))
      BPP_FAIL(BPPGPU_E_INVALID, "model slot %d of node %d out of range", slot_of_node[n], n);
    e->h_branch_model[(size_t)point * e->nn + n] = n == e->root ? 0 : slot_of_node[n];
  }
  BPP_CUDA(cudaMemcpy(e->d_branch_model + (size_t)point * e->nn, &e->h_branch_model[(size_t)point * e->nn],
                      e->nn * sizeof(int), cudaMemcpyHostToDevice));
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_set_branch_lengths(bppgpu_engine* e, int32_t point, const double* t) {
  ENGINE_SYNC(e);
  if (point < 0 || point >= e->npoints || !t) BPP_FAIL(BPPGPU_E_INVALID, "bad point or null array");
  std::copy(t, t + e->nn, e->h_brlen.begin() + (size_t)point * e->nn);
  e->h_brlen[(size_t)point * e->nn + e->root] = 0.0;  // the root has no branch: its table slot is the identity
  // the device copy is refreshed by the next evaluation, ONE transfer for all the points that changed (a batched-points
  // optimiser sets thousands of points per step: a copy + synchronisation per point was 60 ms of its end-to-end step)
  if (e->brlen_dirty_hi <= e->brlen_dirty_lo) { e->brlen_dirty_lo = point; e->brlen_dirty_hi = point + 1; }
  else { e->brlen_dirty_lo = std::min(e->brlen_dirty_lo, (int)point); e->brlen_dirty_hi = std::max(e->brlen_dirty_hi, (int)point + 1); }
  e->have_brlen[point] = 1;
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_set_root_freqs(bppgpu_engine* e, int32_t point, const double* pi) {
  ENGINE_SYNC(e);
  if (point < 0 || point >= e->npoints || !pi) BPP_FAIL(BPPGPU_E_INVALID, "bad point or null array");
  BPP_CUDA(cudaMemcpyAsync(e->d_rootfreq + (size_t)point * e->S, pi, e->S * 8, cudaMemcpyHostToDevice, e->stream));
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  e->have_rootfreq[point] = 1;
  e->rootfreq_used_stale = true;
  e->last_point = -1;
  return BPPGPU_OK;
}

// ---- evaluation ---------------------------------------------------------------------------
static int check_ready(bppgpu_engine* e) {
  if (!e->have_weights) BPP_FAIL(BPPGPU_E_STATE, "pattern weights not set");
  if (!e->have_rates) BPP_FAIL(BPPGPU_E_STATE, "rate classes not set");
  for (int l = 0; l < e->nl; ++l)
    if (!e->have_tip[l]) BPP_FAIL(BPPGPU_E_STATE, "tip codes of leaf node %d not set", e->leaf_nodes[l]);
  for (int p = 0; p < e->npoints; ++p) {
    if (!e->have_brlen[p]) BPP_FAIL(BPPGPU_E_STATE, "branch lengths of point %d not set", p);
    if (!e->have_rootfreq[p] && !(e->flags & BPPGPU_FLAG_WEIGHTED_ROOT))
      BPP_FAIL(BPPGPU_E_STATE, "root frequencies of point %d not set", p);
  }
  std::vector<char> used(e->nmodels, 0);
  e->homogeneous_points = true;
  for (int p = 0; p < e->npoints; ++p) {
    const int first = e->h_branch_model[(size_t)p * e->nn + (e->root == 0 ? 1 : 0)];
    for (int n = 0; n < e->nn; ++n)
      if (n != e->root) {
        used[e->h_branch_model[(size_t)p * e->nn + n]] = 1;
        if (e->h_branch_model[(size_t)p * e->nn + n] != first) e->homogeneous_points = false;
      }
  }
  for (int m = 0; m < e->nmodels; ++m)
    if (used[m] && !e->models[m].set) BPP_FAIL(BPPGPU_E_STATE, "model slot %d is used by a branch but not set", m);
  return BPPGPU_OK;
}

static int ensure_deriv_buffers(bppgpu_engine* e, unsigned want) {
  const size_t tab = (size_t)e->pchunk * e->nn * e->C * e->S * e->S;
  if ((want & (BPPGPU_EVAL_D1 | BPPGPU_EVAL_D2)) && !e->d_dP) BPP_CUDA(dev_alloc(e, &e->d_dP, tab));
  if ((want & BPPGPU_EVAL_D2) && !e->d_d2P) BPP_CUDA(dev_alloc(e, &e->d_d2P, tab));
  if ((want & (BPPGPU_EVAL_D1 | BPPGPU_EVAL_D2)) && !e->d_upper) {
    const size_t clv = (size_t)e->N * e->C * e->S;
    // upper CLVs of tips are read by nobody on the DMMA path: keep them only while they are cheap (accessors/tests)
    const bool all = e->path != PATH_DMMA || (double)e->nn * clv * 8 < 4e9;
    e->upper_slab.assign(e->nn, -1);
    e->n_upper_slabs = 0;
    for (int n = 0; n < e->nn; ++n)
      if (n != e->root && (all || e->leaf_slot[n] < 0)) e->upper_slab[n] = e->n_upper_slabs++;
    BPP_CUDA(dev_alloc(e, &e->d_upper, (size_t)e->n_upper_slabs * clv));
    BPP_CUDA(dev_alloc(e, &e->d_upper_exp, (size_t)e->n_upper_slabs * e->N * e->C));
    if (e->path == PATH_DMMA) {
      const size_t tt = (size_t)e->pchunk * e->nl * e->C * e->ncodes * e->S;
      BPP_CUDA(dev_alloc(e, &e->d_dtiptab, tt));
      BPP_CUDA(dev_alloc(e, &e->d_d2tiptab, tt));
      BPP_CUDA(dev_alloc(e, &e->d_dLc, (size_t)e->N * e->C * 2));
      // per-father fused pass (S = 20): every father with <= 3 sons
      if (e->family) {
        e->fam_mask.assign(e->nn, 0);
        for (int f = 0; f < e->nn; ++f) {
          const int k = e->child_off[f + 1] - e->child_off[f];
          if (k >= 1 && k <= kFamMaxSons)
            for (int j = e->child_off[f]; j < e->child_off[f + 1]; ++j) e->fam_mask[e->children[j]] = 1;
        }
        BPP_CUDA(dev_alloc(e, &e->d_fam_mask, (size_t)e->nn));
        BPP_CUDA(cudaMemcpy(e->d_fam_mask, e->fam_mask.data(), e->nn * sizeof(int), cudaMemcpyHostToDevice));
        {
          auto attr = [](auto k, size_t smem) { return cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); };
          BPP_CUDA(attr(dmma_family_kernel<5, 0>, dmma_family_smem<0>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<5, 0>, dmma_family_smem<0>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<5, 1>, dmma_family_smem<1>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<5, 1>, dmma_family_smem<1>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<5, 2>, dmma_family_smem<2>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<5, 2>, dmma_family_smem<2>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<5, 3>, dmma_family_smem<3>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<5, 3>, dmma_family_smem<3>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<5, 4>, dmma_family_smem<4>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<5, 4>, dmma_family_smem<4>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<8, 0>, dmma_family_smem<0>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<8, 0>, dmma_family_smem<0>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<8, 1>, dmma_family_smem<1>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<8, 1>, dmma_family_smem<1>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<8, 2>, dmma_family_smem<2>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<8, 2>, dmma_family_smem<2>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<8, 3>, dmma_family_smem<3>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<8, 3>, dmma_family_smem<3>(e->C)));
          BPP_CUDA(attr(dmma_family_kernel<8, 4>, dmma_family_smem<4>(e->C)));
          BPP_CUDA(attr(dmma_family_level_kernel<8, 4>, dmma_family_smem<4>(e->C)));
        }
        BPP_CUDA(dev_alloc(e, &e->d_fam_part, (size_t)e->nn * 2 * e->fam_grid));
        BPP_CUDA(cudaMemset(e->d_fam_part, 0, (size_t)e->nn * 2 * e->fam_grid * 8));
        BPP_CUDA(dev_alloc(e, &e->d_fam_packA, (size_t)e->nn * e->C * kFamPackA));
        BPP_CUDA(dev_alloc(e, &e->d_fam_packS, (size_t)e->nn * e->C * kFamPackS));
        BPP_CUDA(dev_alloc(e, &e->d_fam_packT, (size_t)e->nl * e->C * e->ncodes * 64));
      }
    }
  }
  return BPPGPU_OK;
}

static int ensure_scratch(bppgpu_engine* e, bool series, bool chrd) {
  if (!series && !chrd) return BPPGPU_OK;
  const size_t need = (size_t)e->pchunk * e->nn * e->C * e->S * e->S * (series ? 4 : 1);
  if (e->scratch_elems < need) {
    BPP_CUDA(cudaStreamSynchronize(e->stream));
    cudaFree(e->d_scratch);
    e->d_scratch = nullptr;
    BPP_CUDA(dev_alloc(e, &e->d_scratch, need));
    e->scratch_elems = need;
  }
  return BPPGPU_OK;
}

template <int CL, int PT, bool KEEP>
static int walk4_launch_one(const Walk4Params* wp, int grid, size_t smem, cudaStream_t st, bool attr_only) {
  if (attr_only) {
    BPP_CUDA(cudaFuncSetAttribute(walk4_kernel<CL, PT, KEEP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return BPPGPU_OK;
  }
  walk4_kernel<CL, PT, KEEP><<<grid, kWalk4Threads, smem, st>>>(*wp);
  return BPPGPU_OK;
}
template <int CL, int PT>
static int walk4_launch_k(bool keep, const Walk4Params* wp, int grid, size_t smem, cudaStream_t st, bool attr_only) {
  return keep ? walk4_launch_one<CL, PT, true>(wp, grid, smem, st, attr_only)
              : walk4_launch_one<CL, PT, false>(wp, grid, smem, st, attr_only);
}
template <int CL>
static int walk4_launch_pt(int pt, bool keep, const Walk4Params* wp, int grid, size_t smem, cudaStream_t st, bool attr_only) {
  if (pt == 4) return walk4_launch_k<CL, 4>(keep, wp, grid, smem, st, attr_only);
  if (pt == 3) return walk4_launch_k<CL, 3>(keep, wp, grid, smem, st, attr_only);
  if (pt == 2) return walk4_launch_k<CL, 2>(keep, wp, grid, smem, st, attr_only);
  return walk4_launch_k<CL, 1>(keep, wp, grid, smem, st, attr_only);
}
// launches (or, with attr_only, just opts in to the dynamic shared memory of) the walk4 instantiation of this engine
static int walk4_dispatch(bppgpu_engine* e, const Walk4Params* wp, int grid, size_t /*unused*/, cudaStream_t st, bool attr_only) {
  const size_t smem = (size_t)e->prog.nslots * e->w4_pt * kWalk4Threads * 36;
  switch (ilog2(e->C)) {
    case 0: return walk4_launch_pt<0>(e->w4_pt, e->keep, wp, grid, smem, st, attr_only);
    case 1: return walk4_launch_pt<1>(e->w4_pt, e->keep, wp, grid, smem, st, attr_only);
    case 2: return walk4_launch_pt<2>(e->w4_pt, e->keep, wp, grid, smem, st, attr_only);
    default: return walk4_launch_pt<3>(e->w4_pt, e->keep, wp, grid, smem, st, attr_only);
  }
}
static thread_local const W4cProgram* g_w4c_prog = nullptr;   // the launching engine's program (copied into the launch)
template <int CL, int PT, int NW>
static int walk4c_launch_one(const Walk4cParams* wp, int grid, size_t smem, cudaStream_t st, bool attr_only) {
  if (attr_only) {
    BPP_CUDA(cudaFuncSetAttribute(walk4c_kernel<CL, PT, NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return BPPGPU_OK;
  }
  walk4c_kernel<CL, PT, NW><<<grid, NW * 32, smem, st>>>(*wp, *g_w4c_prog);
  return BPPGPU_OK;
}
template <int CL, int NW>
static int walk4c_launch_pt(int pt, const Walk4cParams* wp, int grid, size_t smem, cudaStream_t st, bool attr_only) {
  if (pt == 4) return walk4c_launch_one<CL, 4, NW>(wp, grid, smem, st, attr_only);
  if (pt == 3) return walk4c_launch_one<CL, 3, NW>(wp, grid, smem, st, attr_only);
  if (pt == 2) return walk4c_launch_one<CL, 2, NW>(wp, grid, smem, st, attr_only);
  return walk4c_launch_one<CL, 1, NW>(wp, grid, smem, st, attr_only);
}
static int walk4c_dispatch(bppgpu_engine* e, int pt, const Walk4cParams* wp, int grid, size_t smem, cudaStream_t st, bool attr_only) {
  g_w4c_prog = &e->w4c_prog;
  if (e->w4c_nw == 4) {
    switch (ilog2(e->C)) {
      case 0: return walk4c_launch_pt<0, 4>(pt, wp, grid, smem, st, attr_only);
      case 1: return walk4c_launch_pt<1, 4>(pt, wp, grid, smem, st, attr_only);
      default: return walk4c_launch_pt<2, 4>(pt, wp, grid, smem, st, attr_only);
    }
  }
  switch (ilog2(e->C)) {
    case 0: return walk4c_launch_pt<0, 8>(pt, wp, grid, smem, st, attr_only);
    case 1: return walk4c_launch_pt<1, 8>(pt, wp, grid, smem, st, attr_only);
    case 2: return walk4c_launch_pt<2, 8>(pt, wp, grid, smem, st, attr_only);
    default: return walk4c_launch_pt<3, 8>(pt, wp, grid, smem, st, attr_only);
  }
}
template <int CL>
static void launch_walkS20(const WalkParams& wp, int grid, size_t smem, cudaStream_t st) {
  walkS_kernel<20, CL><<<grid, kWalkThreads, smem, st>>>(wp);
}

// pruning + root reduction of one point (tables of chunk-local index `pl`)
// S = 20 / 64 pruning pass, one launch per (tree level, kind of sons) instead of one per node (dmma_prune_level_kernel).
// The node descriptors are built once and cached on the device; they only hold addresses inside buffers that live as long as
// the engine (checked by signature).
static int enqueue_prune_levels(bppgpu_engine* e, const double* tiptab, cudaStream_t st) {
  const int S = e->S, C = e->C;
  const long long N = e->N;
  const void* sig[3] = {e->d_keep, tiptab, e->d_fam_packL};
  if (e->prune_groups.empty() || sig[0] != e->prune_nodes_sig[0] || sig[1] != e->prune_nodes_sig[1] || sig[2] != e->prune_nodes_sig[2]) {
    const size_t nops = e->gprog.ops.size();
    // level of a node = height of its subtree (sons first in the post-order program)
    std::vector<int> height(e->nn, 0), kind_of(nops, 0), level_of(nops, 0);
    std::vector<DmmaPruneParams> all(nops);
    for (size_t i = 0; i < nops; ++i) {
      const Op& op = e->gprog.ops[i];
      DmmaPruneParams& pp = all[i];
      pp = DmmaPruneParams{};
      pp.nson = op.nchild;
      int kind = op.nchild == 2 ? 0 : 4, h = 0;
      for (int j = 0; j < op.nchild; ++j) {
        const Child& ch = e->gprog.childs[op.child_begin + j];
        PruneSon& ps = pp.sons[j];
        ps.kind = ch.kind == CHILD_TIP ? CHILD_TIP : CHILD_KEEP;
        ps.node = ch.pnode;
        h = std::max(h, height[ch.pnode] + 1);
        if (ch.kind == CHILD_TIP) {
          ps.codes = (const char*)e->d_codes + (size_t)ch.idx * N * e->code_bytes;
          ps.tt = tiptab + (size_t)ch.idx * C * e->ncodes * S;
          if (kind != 4) kind |= 1 << j;
        } else {
          ps.clv = e->d_keep + (size_t)ch.idx * N * C * S;
          ps.exp = e->d_keep_exp + (size_t)ch.idx * N * C;
        }
      }
      height[op.node] = h;
      kind_of[i] = kind;
      level_of[i] = h;
      pp.S = S; pp.C = C; pp.ncodes = e->ncodes; pp.code_bytes = e->code_bytes;
      pp.prow = e->clv_class_major ? 1 : C;
      pp.crow = e->clv_class_major ? (int)N : 1;
      pp.N = N;
      pp.packL = e->d_fam_packL;
      pp.out = e->d_keep + (size_t)op.keep_idx * N * C * S;
      pp.out_exp = e->d_keep_exp + (size_t)op.keep_idx * N * C;
    }
    std::vector<size_t> order(nops);
    for (size_t i = 0; i < nops; ++i) order[i] = i;
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) {
      return level_of[a] != level_of[b] ? level_of[a] < level_of[b] : kind_of[a] < kind_of[b];
    });
    e->prune_groups.clear();
    std::vector<DmmaPruneParams> sorted(nops);
    const long long G = std::max(1, e->fam_grid);
    // rows a CTA must have for its warps to fill their row rings (8 rows per warp and item, a few items each)
    const long long min_ppc = S > 32 ? 256 : 512;
    for (size_t k = 0; k < nops;) {
      size_t k1 = k;
      while (k1 < nops && level_of[order[k1]] == level_of[order[k]] && kind_of[order[k1]] == kind_of[order[k]]) ++k1;
      const long long n = (long long)(k1 - k);
      // CTAs per node: the count whose last wave is fullest, a launch's fixed cost (operand staging, fill, drain ~ `fixed` rows'
      // worth of time) charged once per wave
      long long best_c = 1;
      double best_cost = 1e300;
      const double fixed = 0.15 * (double)N / (double)G;
      for (long long c = 1; c <= G; ++c) {
        long long ppc = (N + c - 1) / c;
        ppc = std::max<long long>(8, (ppc + 7) / 8 * 8);
        if (c > 1 && ppc < min_ppc) break;
        const long long ctas = n * ((N + ppc - 1) / ppc);
        const long long waves = (ctas + G - 1) / G;
        const double cost = (double)waves * ((double)ppc + fixed);
        if (cost < best_cost * (1.0 - 1e-9)) { best_cost = cost; best_c = c; }
      }
      long long ppc = (N + best_c - 1) / best_c;
      ppc = std::max<long long>(8, (ppc + 7) / 8 * 8);
      const int cpn = (int)((N + ppc - 1) / ppc);
      for (size_t j = k; j < k1; ++j) {
        sorted[j] = all[order[j]];
        sorted[j].ppc = (int)ppc;
      }
      e->prune_groups.push_back({kind_of[order[k]], (int)k, (int)n, cpn});
      k = k1;
    }
    BPP_CUDA(cudaMemcpyAsync(e->d_prune_nodes, sorted.data(), nops * sizeof(DmmaPruneParams), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaStreamSynchronize(st));   // (`sorted` goes out of scope)
    for (int i = 0; i < 3; ++i) e->prune_nodes_sig[i] = sig[i];
  }
  for (const bppgpu_engine::PruneGroup& g : e->prune_groups) {
    const DmmaPruneParams* nodes = e->d_prune_nodes + g.first;
    const unsigned grid = (unsigned)g.count * (unsigned)g.ctas_per_node;
#define BPP_PRUNE_L(Sv, Kv) dmma_prune_level_kernel<Sv, Kv, 0><<<grid, prune_threads(Sv, Kv, 0), dmma_prune_smem<Sv, Kv, 0>(C), st>>>(nodes, g.ctas_per_node)
#define BPP_PRUNE_LK(Kv) if (S == 64) BPP_PRUNE_L(64, Kv); else BPP_PRUNE_L(20, Kv)
    switch (g.kind) {
      case 0: BPP_PRUNE_LK(0); break;
      case 1: BPP_PRUNE_LK(1); break;
      case 2: BPP_PRUNE_LK(2); break;
      case 3: BPP_PRUNE_LK(3); break;
      default: BPP_PRUNE_LK(4); break;
    }
#undef BPP_PRUNE_LK
#undef BPP_PRUNE_L
    e->stats.kernel_launches += 1;
  }
  BPP_CUDA(cudaGetLastError());
  return BPPGPU_OK;
}

static int enqueue_prune(bppgpu_engine* e, int point, int pl, cudaStream_t st) {
  const int S = e->S, C = e->C, nn = e->nn;
  const long long N = e->N;
  const size_t SS = (size_t)S * S;
  const double* P = e->d_P + (size_t)pl * nn * C * SS;
  const double* tiptab = e->d_tiptab + (size_t)pl * e->nl * C * e->ncodes * S;
  const double* rootfreq = e->d_rootfreq_used + (size_t)point * S;
  double* site_lnl = e->d_site_lnl + (size_t)point * N;
  double* out = e->d_out + (size_t)point * (1 + 2 * nn);
  const unsigned rflag = (e->flags & BPPGPU_FLAG_R_SEMANTICS) ? 1u : 0u;
  int nparts = 0;
  if (N == 0) {
    BPP_CUDA(cudaMemsetAsync(out, 0, 8, st));
    return BPPGPU_OK;
  }
  if (e->w4c) {
    Walk4cParams wp{};
    wp.stream = e->d_w4c_stream + (size_t)pl * e->w4c_stream_bytes;
    wp.nchunks = e->w4c_nchunks;
    wp.CH = e->w4c_CH;
    wp.nslots = e->prog4c.nslots;
    wp.ncodes = e->ncodes;
    wp.ntips = (int)e->w4c_tip_order.size();
    wp.wide_codes = e->ncodes * e->ncodes;
    wp.max_tips = e->w4c_max_tips;
    wp.flags = rflag;
    wp.rootfreq = rootfreq;
    wp.probs = e->d_probs;
    wp.weights = e->d_weights;
    wp.SR = e->d_SR;
    wp.rexp = e->d_rexp;
    wp.site_lnl = site_lnl;
    wp.partials = e->d_partials;
    wp.parts_total = 0;
    for (const auto& sg : e->w4c_segs) wp.parts_total += sg.grid;
    wp.done_counter = e->d_w4c_counter;
    wp.lnl_out = out;
    for (const auto& sg : e->w4c_segs) {
      wp.codesC = e->d_codesC + sg.codes_off;
      wp.pat0 = sg.pat0;
      wp.pat_end = sg.pat_end;
      wp.part0 = sg.part0;
      int rc4 = walk4c_dispatch(e, sg.pt, &wp, sg.grid, walk4c_smem_bytes(e->w4c_CH, e->prog4c.nslots, C, sg.pt, e->w4c_nw, e->w4c_max_tips), st, false);
      if (rc4) return rc4;
      nparts += sg.grid;
      e->stats.kernel_launches++;
    }
  } else if (e->path == PATH_WALK4) {
    if (e->flags & BPPGPU_FLAG_WEIGHTED_ROOT)
      BPP_FAIL(BPPGPU_E_INVALID, "BPPGPU_FLAG_WEIGHTED_ROOT is served by the generic path only");
    Walk4Params wp{};
    wp.desc = e->d_w4_desc;
    wp.n_ops = (int)e->prog.ops.size();
    wp.nslots = e->prog.nslots;
    wp.ncodes = e->ncodes;
    wp.tstride = e->w4_tstride;
    wp.flags = rflag;
    wp.N = N;
    wp.stream = e->d_w4_stream + (size_t)pl * e->w4_stream_len;
    wp.codesT = e->d_codesT;
    wp.keep = e->d_keep;
    wp.keep_exp = e->d_keep_exp;
    wp.rootfreq = rootfreq;
    wp.probs = e->d_probs;
    wp.weights = e->d_weights;
    wp.SR = e->d_SR;
    wp.rexp = e->d_rexp;
    wp.site_lnl = site_lnl;
    wp.partials = e->d_partials;
    const long long per_cta = (long long)(kWalk4Threads / C) * e->w4_pt;  // patterns per CTA
    const int grid = (int)((N + per_cta - 1) / per_cta);
    nparts = grid;
    int rc4 = walk4_dispatch(e, &wp, grid, 0, st, false);
    if (rc4) return rc4;
    e->stats.kernel_launches++;
  } else if (e->path == PATH_WALKS) {
    if (e->flags & BPPGPU_FLAG_WEIGHTED_ROOT)
      BPP_FAIL(BPPGPU_E_INVALID, "BPPGPU_FLAG_WEIGHTED_ROOT is served by the generic path only");
    WalkParams wp{};
    wp.ops = e->prog.d_ops;
    wp.childs = e->prog.d_childs;
    wp.n_ops = (int)e->prog.ops.size();
    wp.C = C;
    wp.ncodes = e->ncodes;
    wp.code_bytes = e->code_bytes;
    wp.nslots = e->prog.nslots;
    wp.flags = rflag;
    wp.N = N;
    wp.P = P;
    wp.tiptab = tiptab;
    wp.codes = e->d_codes;
    wp.keep = e->d_keep;
    wp.keep_exp = e->d_keep_exp;
    wp.gstack = e->d_gstack;
    wp.gstack_exp = e->d_gstack_exp;
    wp.rootfreq = rootfreq;
    wp.probs = e->d_probs;
    wp.weights = e->d_weights;
    wp.SR = e->d_SR;
    wp.rexp = e->d_rexp;
    wp.site_lnl = site_lnl;
    wp.partials = e->d_partials;
    const long long rows = N * C;
    const int grid = (int)((rows + kWalkThreads - 1) / kWalkThreads);
    nparts = grid;
    const int cl = ilog2(C);
    {
      const size_t smem = (size_t)kMaxStagedChildren * C * (S * S + 2) * 8;
      if (cl == 0) launch_walkS20<0>(wp, grid, smem, st);
      else if (cl == 1) launch_walkS20<1>(wp, grid, smem, st);
      else if (cl == 2) launch_walkS20<2>(wp, grid, smem, st);
      else launch_walkS20<3>(wp, grid, smem, st);
    }
    e->stats.kernel_launches++;
  } else {
    const long long total = N * C * S;
    const int grid_e = (int)std::min<long long>((total + 255) / 256, (long long)g_sm_count * 32);
    const int grid_p = (int)((N + 255) / 256);
    const int grid_r = (int)((N * C + 255) / 256);
    bool prev_chained = false;
    const bool by_level = e->level_batch && e->path == PATH_DMMA && (e->family || e->prune64) && pl == 0;
    if (by_level) {
      int rcl = enqueue_prune_levels(e, tiptab, st);
      if (rcl) return rcl;
    }
    for (const Op& op : e->gprog.ops) {
      if (by_level) break;
      GenericParams gp{};
      gp.childs = e->gprog.d_childs + op.child_begin;
      gp.nchild = op.nchild;
      gp.out_idx = op.keep_idx;
      gp.S = S; gp.C = C; gp.ncodes = e->ncodes; gp.code_bytes = e->code_bytes;
      gp.N = N;
      gp.P = P; gp.tiptab = tiptab; gp.codes = e->d_codes;
      gp.keep = e->d_keep; gp.keep_exp = e->d_keep_exp;
      if (e->path == PATH_DMMA && (e->family || e->prune64) && op.nchild <= kFamMaxSons) {
        DmmaPruneParams pp{};
        pp.nson = op.nchild;
        int kind = op.nchild == 2 ? 0 : 4;
        for (int j = 0; j < op.nchild; ++j) {
          const Child& ch = e->gprog.childs[op.child_begin + j];
          PruneSon& ps = pp.sons[j];
          ps.kind = ch.kind == CHILD_TIP ? CHILD_TIP : CHILD_KEEP;
          ps.node = ch.pnode;
          if (ch.kind == CHILD_TIP) {
            ps.codes = (const char*)e->d_codes + (size_t)ch.idx * N * e->code_bytes;
            ps.tt = tiptab + (size_t)ch.idx * C * e->ncodes * S;
            if (kind != 4) kind |= 1 << j;
          } else {
            ps.clv = e->d_keep + (size_t)ch.idx * N * C * S;
            ps.exp = e->d_keep_exp + (size_t)ch.idx * N * C;
          }
        }
        pp.S = S; pp.C = C; pp.ncodes = e->ncodes; pp.code_bytes = e->code_bytes;
        pp.ppc = e->fam_ppc;
        pp.prow = e->clv_class_major ? 1 : C;
        pp.crow = e->clv_class_major ? (int)N : 1;
        pp.N = N;
        pp.packL = e->d_fam_packL;
        pp.out = e->d_keep + (size_t)op.keep_idx * N * C * S;
        pp.out_exp = e->d_keep_exp + (size_t)op.keep_idx * N * C;
        const int G = e->fam_grid;
        const bool chained = prev_chained;   // the previous launch of this loop was one of these kernels (it calls pdl_wait itself)
        prev_chained = true;
        switch (kind) {
#define BPP_PRUNE(Sv, Kv, Cv) BPP_CUDA(launch_node_kernel(dmma_prune_kernel<Sv, Kv, Cv>, G, prune_threads(Sv, Kv, Cv), dmma_prune_smem<Sv, Kv, Cv>(C), st, chained, pp))
#define BPP_PRUNE_K(Kv) if (S == 64) BPP_PRUNE(64, Kv, 0); else if (e->prune_cfg == 0) BPP_PRUNE(20, Kv, 0); \
                        else if (e->prune_cfg == 1) BPP_PRUNE(20, Kv, 1); else BPP_PRUNE(20, Kv, 2)
          case 0: BPP_PRUNE_K(0); break;
          case 1: BPP_PRUNE_K(1); break;
          case 2: BPP_PRUNE_K(2); break;
          case 3: BPP_PRUNE_K(3); break;
          default: if (S == 64) BPP_PRUNE(64, 4, 0); else BPP_PRUNE(20, 4, 0); break;
#undef BPP_PRUNE_K
#undef BPP_PRUNE
        }
        e->stats.kernel_launches += 1;
      } else if (e->path == PATH_DMMA) {
        DmmaNodeParams dp{};
        dp.childs = gp.childs; dp.nchild = gp.nchild; dp.out_idx = gp.out_idx;
        dp.S = S; dp.C = C; dp.ncodes = e->ncodes; dp.code_bytes = e->code_bytes; dp.N = N;
        dp.P = P; dp.tiptab = tiptab; dp.codes = e->d_codes; dp.keep = e->d_keep; dp.keep_exp = e->d_keep_exp;
        int nint = 0;
        for (int j = 0; j < op.nchild; ++j)
          if (e->gprog.childs[op.child_begin + j].kind != CHILD_TIP) ++nint;
        static const int rw_env = getenv("BPPGPU_DMMA_RW") ? atoi(getenv("BPPGPU_DMMA_RW")) : 0;   // tuning knob
        static const int cta_env = getenv("BPPGPU_DMMA_CTAS") ? atoi(getenv("BPPGPU_DMMA_CTAS")) : 0;
        auto launch = [&](auto kern, int RW, size_t smem, int ctas_per_sm) {
          const long long tiles = (N + 8 * RW * kDmmaNodeWarps - 1) / (8 * RW * kDmmaNodeWarps);
          if (cta_env > 0) ctas_per_sm = cta_env;
          const dim3 grid((unsigned)std::min<long long>(tiles, std::max(1, g_sm_count * ctas_per_sm / C)), (unsigned)C);
          kern<<<grid, kDmmaNodeWarps * 32, smem, st>>>(dp);
        };
        prev_chained = false;
        if (S <= 20) {
          const size_t smem = nint * dmma_node_smem_per_child<5, 3>();
          if (rw_env == 1) launch(dmma_node_kernel<5, 3, 1>, 1, smem, 12);
          else if (rw_env == 4) launch(dmma_node_kernel<5, 3, 4>, 4, smem, 4);
          else launch(dmma_node_kernel<5, 3, 2>, 2, smem, 8);
        } else {
          const size_t smem = nint * dmma_node_smem_per_child<16, 8>();
          if (rw_env == 2) launch(dmma_node_kernel<16, 8, 2>, 2, smem, 2);
          else launch(dmma_node_kernel<16, 8, 1>, 1, smem, 2);
        }
        e->stats.kernel_launches += 1;
      } else {
        generic_node_kernel<<<grid_e, 256, 0, st>>>(gp);
        generic_scale_kernel<<<grid_r, 256, 0, st>>>(gp);
        prev_chained = false;
        e->stats.kernel_launches += 2;
      }
    }
    const int ridx = e->internal_idx[e->root];
    if (e->flags & BPPGPU_FLAG_WEIGHTED_ROOT) {
      WeightedRootParams wr{};
      wr.root_clv = e->d_keep + (size_t)ridx * N * C * S;
      wr.root_exp = e->d_keep_exp + (size_t)ridx * N * C;
      wr.S = S; wr.C = C; wr.N = N;
      wr.probs = e->d_probs;
      wr.out = e->d_rootfreq_used + (size_t)point * S;
      // partial record of this shard, exchanged between the GPUs of the job (one all-gather of S + 1 doubles), combined
      weighted_root_partial_kernel<<<1, 256, 0, st>>>(wr, e->d_wr_recs + (size_t)e->comm_rank * (S + 1));
      if (e->comm && e->comm_nranks > 1)
        BPP_NCCL(nccl_api().AllGather(e->d_wr_recs + (size_t)e->comm_rank * (S + 1), e->d_wr_recs, (size_t)(S + 1), ncclDouble,
                                      (ncclComm_t)e->comm, st));
      weighted_root_combine_kernel<<<1, 256, 0, st>>>(e->d_wr_recs, e->comm_nranks, S, wr.out);
      e->stats.kernel_launches += 2;
    }
    RootParams rp{};
    rp.root_clv = e->d_keep + (size_t)ridx * N * C * S;
    rp.root_exp = e->d_keep_exp + (size_t)ridx * N * C;
    rp.S = S; rp.C = C; rp.flags = rflag; rp.N = N;
    rp.prow = e->clv_class_major ? 1 : C;
    rp.crow = e->clv_class_major ? N : 1;
    rp.rootfreq = rootfreq; rp.probs = e->d_probs; rp.weights = e->d_weights;
    rp.SR = e->d_SR; rp.rexp = e->d_rexp; rp.site_lnl = site_lnl; rp.partials = e->d_partials;
    generic_root_kernel<<<grid_p, 256, 0, st>>>(rp);
    e->stats.kernel_launches++;
    nparts = grid_p;
  }
  if (!e->w4c) {   // (the chunk-streamed walk adds its partials up itself)
    finalize_sum_kernel<<<1, 256, 0, st>>>(e->d_partials, nparts, out);
    e->stats.kernel_launches++;
  }
  BPP_CUDA(cudaGetLastError());
  long long upd = 0;
  for (const Op& op : e->prog.ops) (void)op, upd += N * C * S;
  e->stats.clv_updates += upd;
  return BPPGPU_OK;
}

// prefix pass + derivatives for one point, generic kernels (lower CLVs must be resident)
static int enqueue_derivs(bppgpu_engine* e, int point, int pl, unsigned want, cudaStream_t st) {
  const int S = e->S, C = e->C, nn = e->nn;
  const long long N = e->N;
  const size_t SS = (size_t)S * S;
  const size_t clv = (size_t)N * C * S;
  const double* P = e->d_P + (size_t)pl * nn * C * SS;
  const double* dP = e->d_dP + (size_t)pl * nn * C * SS;
  const double* d2P = (want & BPPGPU_EVAL_D2) ? e->d_d2P + (size_t)pl * nn * C * SS : nullptr;
  const double* tiptab = e->d_tiptab + (size_t)pl * e->nl * C * e->ncodes * S;
  double* out = e->d_out + (size_t)point * (1 + 2 * nn);
  if (N == 0) return BPPGPU_OK;
  const long long total = N * C * S;
  const int grid_e = (int)std::min<long long>((total + 255) / 256, (long long)g_sm_count * 32);
  const int grid_p = (int)((N + 255) / 256);
  const int grid_r = (int)((N * C + 255) / 256);
  const bool family = e->path == PATH_DMMA && e->family;
  bool prev_family = false;   // the previous launch was a dmma_family_kernel (programmatic dependent launch chain)
  cudaError_t fam_err = cudaSuccess;
  auto build_family = [&](int f, int* kind_out) {
    DmmaFamilyParams fp{};
    const size_t clvN = (size_t)N * C * S, expN = (size_t)N * C;
    fp.nson = e->child_off[f + 1] - e->child_off[f];
    int kind = fp.nson == 2 ? 0 : 4;
    for (int j = 0; j < fp.nson; ++j) {
      const int s = e->children[e->child_off[f] + j];
      const bool tip = e->leaf_slot[s] >= 0;
      FamilySon& fs = fp.sons[j];
      fs.kind = tip ? CHILD_TIP : CHILD_KEEP;
      fs.node = s;
      if (tip) {
        const int slot = e->leaf_slot[s];
        fs.codes = (const char*)e->d_codes + (size_t)slot * N * e->code_bytes;
        fs.tpack = e->d_fam_packT + (size_t)slot * C * e->ncodes * 64;
        if (kind != 4) kind |= 1 << j;
      } else {
        fs.clv = e->d_keep + (size_t)e->internal_idx[s] * clvN;
        fs.exp = e->d_keep_exp + (size_t)e->internal_idx[s] * expN;
      }
      if (e->upper_slab[s] >= 0) {
        fs.up = e->d_upper + (size_t)e->upper_slab[s] * clvN;
        fs.upexp = e->d_upper_exp + (size_t)e->upper_slab[s] * expN;
      }
    }
    fp.father = f == e->root ? -1 : f;
    if (f != e->root) {
      fp.fup = e->d_upper + (size_t)e->upper_slab[f] * clvN;
      fp.fupexp = e->d_upper_exp + (size_t)e->upper_slab[f] * expN;
    }
    fp.S = S; fp.C = C; fp.ncodes = e->ncodes; fp.code_bytes = e->code_bytes;
    fp.nh_form = (e->flags & BPPGPU_FLAG_NH_DERIV) ? 1 : 0;
    fp.ppc = e->fam_ppc;
    fp.prow = e->clv_class_major ? 1 : C;
    fp.crow = e->clv_class_major ? (int)N : 1;
    fp.N = N;
    fp.packA = e->d_fam_packA; fp.packS = e->d_fam_packS;
    fp.rootfreq = e->d_rootfreq_used + (size_t)point * S;
    fp.probs = e->d_probs; fp.SR = e->d_SR; fp.weights = e->d_weights; fp.rexp = e->d_rexp;
    fp.part = e->d_fam_part;
    fp.part_stride = e->fam_grid;
    *kind_out = kind;
    return fp;
  };
  auto launch_family = [&](int f) {
    int kind = 0;
    const DmmaFamilyParams fp = build_family(f, &kind);
    const bool d2 = (want & BPPGPU_EVAL_D2) != 0;
    const int G = e->fam_grid;
    const bool fam_chained = prev_family;
    prev_family = true;
#define BPP_FAM(NBv, Kv) fam_err = launch_node_kernel(dmma_family_kernel<NBv, Kv>, G, fam_threads_kind(Kv), dmma_family_smem<Kv>(C), st, fam_chained, fp)
    switch (kind) {
      case 0: if (d2) BPP_FAM(8, 0); else BPP_FAM(5, 0); break;
      case 1: if (d2) BPP_FAM(8, 1); else BPP_FAM(5, 1); break;
      case 2: if (d2) BPP_FAM(8, 2); else BPP_FAM(5, 2); break;
      case 3: if (d2) BPP_FAM(8, 3); else BPP_FAM(5, 3); break;
      default: if (d2) BPP_FAM(8, 4); else BPP_FAM(5, 4); break;
    }
#undef BPP_FAM
    e->stats.kernel_launches++;
  };
  auto launch_branch = [&](int n) {
    prev_family = false;
    const int f = e->parent[n];
    UpperParams up{};
    up.sibs = e->d_sibs + e->sib_off[n];
    up.nsib = e->sib_off[n + 1] - e->sib_off[n];
    up.father = f == e->root ? -1 : f;
    up.S = S; up.C = C; up.ncodes = e->ncodes; up.code_bytes = e->code_bytes;
    up.N = N;
    up.P = P; up.tiptab = tiptab; up.codes = e->d_codes;
    up.keep = e->d_keep; up.keep_exp = e->d_keep_exp;
    const int fslab = f == e->root ? 0 : e->upper_slab[f];
    const int nslab = e->upper_slab[n];
    if (e->path == PATH_DMMA) {
      DmmaUpperParams du{};
      du.sibs = e->d_sibs + e->sib_off[n];
      du.nsib = e->sib_off[n + 1] - e->sib_off[n];
      du.father = f == e->root ? -1 : f;
      du.father_upper = fslab;
      du.node = n;
      du.node_is_tip = e->leaf_slot[n] >= 0;
      du.node_idx = du.node_is_tip ? e->leaf_slot[n] : e->internal_idx[n];
      du.upper_out = nslab;
      du.S = S; du.C = C; du.ncodes = e->ncodes; du.code_bytes = e->code_bytes;
      du.nh_form = (e->flags & BPPGPU_FLAG_NH_DERIV) ? 1 : 0;
      du.want = want;
      du.N = N;
      du.P = P; du.dP = dP; du.d2P = d2P;
      du.tiptab = tiptab;
      du.dtiptab = e->d_dtiptab + (size_t)pl * e->nl * C * e->ncodes * S;
      du.d2tiptab = e->d_d2tiptab + (size_t)pl * e->nl * C * e->ncodes * S;
      du.codes = e->d_codes;
      du.keep = e->d_keep; du.keep_exp = e->d_keep_exp;
      du.upper = e->d_upper; du.upper_exp = e->d_upper_exp;
      du.rootfreq = e->d_rootfreq_used + (size_t)point * S;
      du.probs = e->d_probs; du.SR = e->d_SR; du.rexp = e->d_rexp;
      du.dLc = e->d_dLc;
      int nmat = (du.father >= 0 ? 1 : 0);
      for (int k = e->sib_off[n]; k < e->sib_off[n + 1]; ++k)
        if (e->sibs_flat[k].kind != CHILD_TIP) ++nmat;
      if (!du.node_is_tip) nmat += ((want & 2u) ? 1 : 0) + ((want & 4u) ? 1 : 0) + du.nh_form;
      static const int drw_env = getenv("BPPGPU_DERIV_RW") ? atoi(getenv("BPPGPU_DERIV_RW")) : 0;   // tuning knob
      auto launch = [&](auto kern, int RW, size_t smem, int ctas_per_sm) {
        const long long tiles = (N + 8 * RW * kDmmaNodeWarps - 1) / (8 * RW * kDmmaNodeWarps);
        const dim3 grid((unsigned)std::min<long long>(tiles, std::max(1, g_sm_count * ctas_per_sm / C)), (unsigned)C);
        kern<<<grid, kDmmaNodeWarps * 32, smem, st>>>(du);
      };
      if (S <= 20) {
        const size_t smem = nmat * dmma_node_smem_per_child<5, 3>();
        if (drw_env == 2) launch(dmma_upper_deriv_kernel<5, 3, 2>, 2, smem, 8);
        else launch(dmma_upper_deriv_kernel<5, 3, 1>, 1, smem, 16);
      } else {
        launch(dmma_upper_deriv_kernel<16, 8, 1>, 1, nmat * dmma_node_smem_per_child<16, 8>(), 4);
      }
      deriv_combine_kernel<<<grid_p, 256, 0, st>>>(e->d_dLc, e->d_weights, C, N, e->d_partials, e->d_partials2);
      finalize_sum2_kernel<<<1, 256, 0, st>>>(e->d_partials, e->d_partials2, grid_p, out + 1 + n, out + 1 + nn + n);
      e->stats.kernel_launches += 3;
      return;
    }
    up.upper_f = e->d_upper + (size_t)fslab * clv;
    up.uexp_f = e->d_upper_exp + (size_t)fslab * N * C;
    up.rootfreq = e->d_rootfreq_used + (size_t)point * S;
    up.upper_out = e->d_upper + (size_t)nslab * clv;
    up.uexp_out = e->d_upper_exp + (size_t)nslab * N * C;
    upper_node_kernel<<<grid_e, 256, 0, st>>>(up);
    upper_scale_kernel<<<grid_r, 256, 0, st>>>(up);
    DerivParams dp{};
    dp.node = n;
    dp.is_tip = e->leaf_slot[n] >= 0;
    dp.idx = dp.is_tip ? e->leaf_slot[n] : e->internal_idx[n];
    dp.S = S; dp.C = C; dp.code_bytes = e->code_bytes;
    dp.nh_form = (e->flags & BPPGPU_FLAG_NH_DERIV) ? 1 : 0;
    dp.want = want;
    dp.N = N;
    dp.P = P + (size_t)n * C * SS;
    dp.dP = dP + (size_t)n * C * SS;
    dp.d2P = d2P ? d2P + (size_t)n * C * SS : nullptr;
    dp.code_table = e->d_code_table;
    dp.codes = e->d_codes;
    dp.keep = e->d_keep; dp.keep_exp = e->d_keep_exp;
    dp.upper = up.upper_out; dp.uexp = up.uexp_out;
    dp.SR = e->d_SR; dp.rexp = e->d_rexp;
    dp.probs = e->d_probs; dp.weights = e->d_weights;
    dp.part1 = e->d_partials; dp.part2 = e->d_partials2;
    deriv_node_kernel<<<grid_p, 256, 0, st>>>(dp);
    finalize_sum_kernel<<<1, 256, 0, st>>>(e->d_partials, grid_p, out + 1 + n);
    finalize_sum_kernel<<<1, 256, 0, st>>>(e->d_partials2, grid_p, out + 1 + nn + n);
    e->stats.kernel_launches += 5;
  };
  // one launch per (depth, kind of sons) when every father is within the family kernel's son limit (dmma_family_level_kernel)
  // (measured on cfg3: 73.6 ms against 70.9 ms for one launch per father -- the derivative launches are long enough (140 us) that
  //  their fixed cost does not matter, so this stays opt-in; the pruning pass, 54 us per launch, gains 8-13 %)
  const bool deriv_levels = getenv("BPPGPU_LEVEL_BATCH_DERIV") && atoi(getenv("BPPGPU_LEVEL_BATCH_DERIV")) != 0;
  const bool by_level = deriv_levels && family && e->level_batch && pl == 0 && e->d_family_nodes != nullptr;
  if (by_level) {
    const void* sig[4] = {e->d_keep, e->d_upper, e->d_fam_packS, e->d_fam_part};
    const unsigned wsig = (want & BPPGPU_EVAL_D2) | ((e->flags & BPPGPU_FLAG_NH_DERIV) ? 0x100u : 0u) | 0x1000u;
    if (e->family_groups.empty() || memcmp(sig, e->family_nodes_sig, sizeof(sig)) != 0 || wsig != e->family_nodes_want) {
      std::vector<int> depth(nn, 0), fathers, kinds;
      for (int n : e->preorder) {
        if (n != e->root) depth[n] = depth[e->parent[n]] + 1;
        if (e->child_off[n + 1] - e->child_off[n] >= 1) fathers.push_back(n);
      }
      std::vector<DmmaFamilyParams> all(fathers.size());
      kinds.resize(fathers.size());
      for (size_t i = 0; i < fathers.size(); ++i) all[i] = build_family(fathers[i], &kinds[i]);
      std::vector<size_t> order(fathers.size());
      for (size_t i = 0; i < order.size(); ++i) order[i] = i;
      std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) {
        return depth[fathers[a]] != depth[fathers[b]] ? depth[fathers[a]] < depth[fathers[b]] : kinds[a] < kinds[b];
      });
      e->family_groups.clear();
      std::vector<DmmaFamilyParams> sorted(fathers.size());
      const long long G = std::max(1, e->fam_grid);
      const double fixed = 0.15 * (double)N / (double)G;
      for (size_t k = 0; k < order.size();) {
        size_t k1 = k;
        while (k1 < order.size() && depth[fathers[order[k1]]] == depth[fathers[order[k]]] && kinds[order[k1]] == kinds[order[k]]) ++k1;
        const long long n = (long long)(k1 - k);
        long long best_c = 1;
        double best_cost = 1e300;
        for (long long c = 1; c <= G; ++c) {
          long long ppc = std::max<long long>(8, ((N + c - 1) / c + 7) / 8 * 8);
          if (c > 1 && ppc < 384) break;
          const long long waves = (n * ((N + ppc - 1) / ppc) + G - 1) / G;
          const double cost = (double)waves * ((double)ppc + fixed);
          if (cost < best_cost * (1.0 - 1e-9)) { best_cost = cost; best_c = c; }
        }
        const long long ppc = std::max<long long>(8, ((N + best_c - 1) / best_c + 7) / 8 * 8);
        for (size_t j = k; j < k1; ++j) {
          sorted[j] = all[order[j]];
          sorted[j].ppc = (int)ppc;
        }
        e->family_groups.push_back({kinds[order[k]], (int)k, (int)n, (int)((N + ppc - 1) / ppc)});
        k = k1;
      }
      BPP_CUDA(cudaMemcpyAsync(e->d_family_nodes, sorted.data(), sorted.size() * sizeof(DmmaFamilyParams), cudaMemcpyHostToDevice, st));
      BPP_CUDA(cudaStreamSynchronize(st));
      memcpy(e->family_nodes_sig, sig, sizeof(sig));
      e->family_nodes_want = wsig;
    }
    const bool d2 = (want & BPPGPU_EVAL_D2) != 0;
    for (const bppgpu_engine::PruneGroup& g : e->family_groups) {
      const DmmaFamilyParams* fathers = e->d_family_nodes + g.first;
      const unsigned grid = (unsigned)g.count * (unsigned)g.ctas_per_node;
#define BPP_FAM_L(NBv, Kv) dmma_family_level_kernel<NBv, Kv><<<grid, fam_threads_kind(Kv), dmma_family_smem<Kv>(C), st>>>(fathers, g.ctas_per_node)
      switch (g.kind) {
        case 0: if (d2) BPP_FAM_L(8, 0); else BPP_FAM_L(5, 0); break;
        case 1: if (d2) BPP_FAM_L(8, 1); else BPP_FAM_L(5, 1); break;
        case 2: if (d2) BPP_FAM_L(8, 2); else BPP_FAM_L(5, 2); break;
        case 3: if (d2) BPP_FAM_L(8, 3); else BPP_FAM_L(5, 3); break;
        default: if (d2) BPP_FAM_L(8, 4); else BPP_FAM_L(5, 4); break;
      }
#undef BPP_FAM_L
      e->stats.kernel_launches++;
    }
    BPP_CUDA(cudaGetLastError());
  }
  for (int n : e->preorder) {
    if (by_level) break;
    if (n != e->root && !(family && e->fam_mask[n])) launch_branch(n);
    if (family) {
      // the sons of n in one launch (upper[n] is complete: n's own launch precedes this one in pre-order)
      const int k = e->child_off[n + 1] - e->child_off[n];
      if (k >= 1 && k <= kFamMaxSons) launch_family(n);
      BPP_CUDA(fam_err);
    }
  }
  if (family) {
    finalize_family_kernel<<<nn, 128, 0, st>>>(e->d_fam_part, e->d_fam_mask, e->fam_grid, nn, out, want);
    e->stats.kernel_launches++;
  }
  BPP_CUDA(cudaGetLastError());
  return BPPGPU_OK;
}

// table route buffers of a factored engine, allocated the first time the guard sends a point there
static int ensure_tables(bppgpu_engine* e) {
  if (e->tables_allocated) return BPPGPU_OK;
  const int nn = e->nn, S = e->S, C = e->C;
  const size_t SS = (size_t)S * S, per_point = (size_t)nn * C * SS * 8;
  size_t fr = 0, tot = 0;
  if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) fr = (size_t)8 << 30;
  const size_t clv = (size_t)e->N * C * S;
  e->pchunk = (int)std::max<size_t>(1, std::min<size_t>((size_t)e->npoints, (fr / 2) / (5 * per_point + e->ni * clv * 8)));   // + series scratch
  BPP_CUDA(dev_alloc(e, &e->d_P, (size_t)e->pchunk * nn * C * SS));
  BPP_CUDA(dev_alloc(e, &e->d_keep, (size_t)e->pchunk * e->ni * clv));
  BPP_CUDA(dev_alloc(e, &e->d_keep_exp, (size_t)e->pchunk * e->ni * e->N * C));
  e->tables_allocated = true;
  return BPPGPU_OK;
}

// The factored route of a batched-points engine (chr_factored_kernels.cuh): guard, level kernels, root.  `ranges` receives
// the runs of consecutive points that must go through the table route instead (guard failures, singular generators).
static int eval_points_factored(bppgpu_engine* e, cudaStream_t st, bool any_real, bool any_complex,
                                std::vector<std::pair<int, int>>& ranges) {
  const int nn = e->nn, S = e->S, npts = e->npoints;
  const size_t SS = (size_t)S * S;
  // ---- tiles: sons grouped by the height of their subtree, observed tips apart from dense columns -------------------------
  if (e->chr_tiles_dirty) {
    std::vector<int> height(nn, 0), leaf_state(nn, -2);
    std::vector<double> leaf_vec((size_t)nn * S, 0.0);
    for (int k = nn - 1; k >= 0; --k) {   // reverse pre-order: sons first
      const int n = e->preorder[k];
      for (int c = e->child_off[n]; c < e->child_off[n + 1]; ++c) height[n] = std::max(height[n], height[e->children[c]] + 1);
      if (e->leaf_slot[n] >= 0) {
        const int code = e->h_codes[(size_t)e->leaf_slot[n]];
        leaf_state[n] = e->h_code_single[(size_t)code];
        if (leaf_state[n] < 0) {
          leaf_state[n] = -1;
          std::copy(e->h_code_table.begin() + (size_t)code * S, e->h_code_table.begin() + (size_t)(code + 1) * S, leaf_vec.begin() + (size_t)n * S);
        }
      }
    }
    const int hmax = height[e->root];
    std::vector<int> edges, kinds;
    e->chr_level_tile0.assign(1, 0);
    for (int h = 0; h < hmax; ++h) {
      for (int kind = 0; kind < 2; ++kind) {
        std::vector<int> members;
        for (int n = 0; n < nn; ++n) {
          if (n == e->root || height[n] != h) continue;
          const int kd = (e->leaf_slot[n] >= 0 && leaf_state[n] >= 0) ? 0 : 1;
          if (kd == kind) members.push_back(n);
        }
        // observed tips by state: the columns of a tile then gather neighbouring entries of V^-1 (any order within a level is valid)
        if (kind == 0) std::stable_sort(members.begin(), members.end(), [&](int a, int b) { return leaf_state[a] < leaf_state[b]; });
        int fill = 0;
        for (int n : members) {
          if (fill == 0) { edges.resize(edges.size() + kChrCols, -1); kinds.push_back(kind); }
          edges[edges.size() - kChrCols + fill] = n;
          fill = (fill + 1) % kChrCols;
        }
      }
      e->chr_level_tile0.push_back((int)kinds.size());
    }
    e->chr_ntiles = (int)kinds.size();
    e->stats.chr_tiles_tip = (int)std::count(kinds.begin(), kinds.end(), 0);
    e->stats.chr_tiles_dense = (int)std::count(kinds.begin(), kinds.end(), 1);
    e->stats.chr_cblocks_tip = e->stats.chr_cblocks_dense = 0;
    for (size_t t = 0; t < kinds.size(); ++t) {
      int used = 0;
      for (int j = 0; j < kChrCols; ++j) used += edges[t * kChrCols + j] >= 0;
      (kinds[t] == 0 ? e->stats.chr_cblocks_tip : e->stats.chr_cblocks_dense) += (used + 7) / 8;
    }
    BPP_CUDA(cudaMemcpyAsync(e->d_chr_tile_edges, edges.data(), edges.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaMemcpyAsync(e->d_chr_tile_kind, kinds.data(), kinds.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaMemcpyAsync(e->d_chr_leaf_state, leaf_state.data(), nn * sizeof(int), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaMemcpyAsync(e->d_chr_leaf_vec, leaf_vec.data(), leaf_vec.size() * 8, cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaStreamSynchronize(st));   // the host vectors go out of scope
    e->chr_tiles_dirty = false;
  }
  // ---- guard --------------------------------------------------------------------------------------------------------------
  const int probe_node = e->root == 0 ? 1 : 0;
  e->chr_bad.assign(npts, 0);
  static const bool guard_on = !(getenv("BPPGPU_POINTS_GUARD") && atoi(getenv("BPPGPU_POINTS_GUARD")) == 0);
  static const double guard_tol = getenv("BPPGPU_POINTS_GUARD_TOL") ? atof(getenv("BPPGPU_POINTS_GUARD_TOL")) : kChrGuardTol;   // experiments
  std::vector<double> probe_t((size_t)npts * 3);
  std::vector<int> probe_bm((size_t)npts * 3);
  for (int p = 0; p < npts; ++p) {
    const int slot = e->h_branch_model[(size_t)p * nn + probe_node];
    if (!(e->models[slot].flags & BPPGPU_MODEL_NONSINGULAR)) e->chr_bad[p] = 1;
    double tmin = 1e300, tmax = 0.0;
    for (int n = 0; n < nn; ++n) {
      if (n == e->root) continue;
      const double t = e->h_brlen[(size_t)p * nn + n];
      tmin = std::min(tmin, t);
      tmax = std::max(tmax, t);
    }
    if (!(tmin > 0)) tmin = tmax * 1e-3;
    probe_t[(size_t)p * 3] = tmin;
    probe_t[(size_t)p * 3 + 1] = std::sqrt(tmin * tmax);
    probe_t[(size_t)p * 3 + 2] = tmax;
    probe_bm[(size_t)p * 3] = probe_bm[(size_t)p * 3 + 1] = probe_bm[(size_t)p * 3 + 2] = slot;
  }
  BPP_CUDA(cudaEventRecord(e->ptring_a[e->ptring_head], st));
  BPP_CUDA(cudaMemcpyAsync(e->d_chr_bad, e->chr_bad.data(), npts * sizeof(int), cudaMemcpyHostToDevice, st));
  if (guard_on) {
    BPP_CUDA(cudaMemcpyAsync(e->d_chr_probe_t, probe_t.data(), probe_t.size() * 8, cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaMemcpyAsync(e->d_chr_probe_bm, probe_bm.data(), probe_bm.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    std::vector<ModelDev> md(e->nmodels);
    for (int m = 0; m < e->nmodels; ++m) {
      md[m] = to_dev(e->models[m]);
      md[m].flags &= ~(unsigned)BPPGPU_MODEL_CLAMP01;   // the guard looks at the entries BEFORE the reference's clamp
    }
    BPP_CUDA(cudaMemcpyAsync(e->d_models_noclamp, md.data(), md.size() * sizeof(ModelDev), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaStreamSynchronize(st));
    for (int g0 = 0; g0 < npts; g0 += e->gchunk) {
      const int np = std::min(e->gchunk, npts - g0);
      long long launches = 0;
      int rc = launch_pt(st, e->d_models_noclamp, false, false, any_real, any_complex, false, e->d_chr_probe_bm + (size_t)g0 * 3,
                         e->d_chr_probe_t + (size_t)g0 * 3, e->d_rates, S, 1, 3, -1, np, BPPGPU_WANT_P, e->d_chr_guardP, nullptr, nullptr,
                         nullptr, e->d_status, &launches);
      if (rc) return rc;
      chr_guard_kernel<<<np, 256, 0, st>>>(e->d_chr_guardP, 3, S, guard_tol, e->d_chr_bad, g0);
      e->stats.kernel_launches += launches + 1;
    }
    BPP_CUDA(cudaMemcpyAsync(e->chr_bad.data(), e->d_chr_bad, npts * sizeof(int), cudaMemcpyDeviceToHost, st));
    BPP_CUDA(cudaStreamSynchronize(st));
  }
  BPP_CUDA(cudaEventRecord(e->ptring_b[e->ptring_head], st));
  e->ptring_head = (e->ptring_head + 1) % bppgpu_engine::kRing;
  e->ptring_n = std::min(e->ptring_n + 1, (int)bppgpu_engine::kRing);
  // ---- levels + root ------------------------------------------------------------------------------------------------------
  BPP_CUDA(cudaEventRecord(e->ring_a[e->ring_head], st));
  const size_t smem = chr_level_smem(S);
  // slab-streamed kernels: ring depth from the shared memory left beside the column tile -- two CTAs per SM for the level
  // launches (several tiles of a point run side by side), one per SM for the chain (148 resident points' eigenvectors fit in L2)
  int nst_level = 0, nst_chain = 0;
  if (e->chr_slab) {
    const int K8 = (S + 7) & ~7;
    const size_t base = chr_slab_smem(S, 0), slab = (size_t)chr_slab_doubles(K8) * 8;
    static const int lv_env = getenv("BPPGPU_CHR_NST_LEVEL") ? atoi(getenv("BPPGPU_CHR_NST_LEVEL")) : 0;   // tuning knobs
    static const int ch_env = getenv("BPPGPU_CHR_NST_CHAIN") ? atoi(getenv("BPPGPU_CHR_NST_CHAIN")) : 0;
    nst_level = (int)std::min<size_t>(kChrMaxStages, (((size_t)g_smem_per_sm / 2 - 1024) > base ? ((size_t)g_smem_per_sm / 2 - 1024 - base) / slab : 0));
    nst_chain = (int)std::min<size_t>(kChrMaxStages, ((size_t)g_smem_optin > base ? ((size_t)g_smem_optin - base) / slab : 0));
    if (nst_level < 2) nst_level = (int)std::min<size_t>(kChrMaxStages, ((size_t)g_smem_optin > base ? ((size_t)g_smem_optin - base) / slab : 0));
    if (lv_env >= 2) nst_level = std::min(lv_env, nst_chain);
    if (ch_env >= 2) nst_chain = std::min(ch_env, nst_chain);
    if (nst_level < 2 || nst_chain < 2) BPP_FAIL(BPPGPU_E_INVALID, "no room for the slab ring at S = %d", S);
    if (e->chr_slab_dirty) {
      chr_slab_kernel<<<dim3(8, (unsigned)e->nmodels), 256, 0, st>>>(e->d_models, S, K8, e->d_chr_aslab);
      e->stats.kernel_launches++;
      e->chr_slab_dirty = false;
    }
  }
  for (int f0 = 0; f0 < npts; f0 += e->fchunk) {
    const int np = std::min(e->fchunk, npts - f0);
    ChrLevelParams lp{};
    lp.models = e->d_models; lp.branch_model = e->d_branch_model; lp.brlen = e->d_brlen;
    lp.rate0 = e->h_rates[0];
    lp.S = S; lp.nn = nn; lp.p0 = f0;
    lp.tile_edges = e->d_chr_tile_edges; lp.tile_kind = e->d_chr_tile_kind;
    lp.child_off = e->d_child_off; lp.children = e->d_children;
    lp.leaf_state = e->d_chr_leaf_state; lp.leaf_vec = e->d_chr_leaf_vec;
    lp.term = e->d_chr_term; lp.term_exp = e->d_chr_term_exp;
    lp.skip = e->d_chr_bad;
    lp.aslab = e->d_chr_aslab;
    // first level from which every level is one tile: those go in one chain launch (chr_chain_kernel)
    static const bool chain_on = !(getenv("BPPGPU_CHR_CHAIN") && atoi(getenv("BPPGPU_CHR_CHAIN")) == 0);
    const size_t nlev = e->chr_level_tile0.size() - 1;
    size_t chain0 = nlev;
    while (chain_on && chain0 > 0 && e->chr_level_tile0[chain0] - e->chr_level_tile0[chain0 - 1] == 1) --chain0;
    if (nlev - chain0 < 3) chain0 = nlev;   // not worth a different schedule
    for (size_t l = 0; l < chain0; ++l) {
      const int t0 = e->chr_level_tile0[l], nt = e->chr_level_tile0[l + 1] - t0;
      if (nt <= 0) continue;
      lp.tile0 = t0;
      for (int y0 = 0; y0 < np; y0 += 65535) {   // gridDim.y limit
        ChrLevelParams q = lp;
        q.p0 = f0 + y0;
        q.term = e->d_chr_term + (size_t)y0 * nn * S;
        q.term_exp = e->d_chr_term_exp + (size_t)y0 * nn;
        if (e->chr_slab) {
          q.nst = nst_level;
          chr_level_slab_kernel<<<dim3((unsigned)nt, (unsigned)std::min(65535, np - y0)), (kChrCons + 1) * 32, chr_slab_smem(S, nst_level), st>>>(q);
        } else {
          chr_level_kernel<<<dim3((unsigned)nt, (unsigned)std::min(65535, np - y0)), kChrWarps * 32, smem, st>>>(q);
        }
        e->stats.kernel_launches++;
      }
    }
    if (chain0 < nlev) {
      ChrLevelParams q = lp;
      q.tile0 = e->chr_level_tile0[chain0];
      // more than half of an SM's shared memory: one CTA per SM, so that the resident points' eigenvectors fit in L2
      const size_t chain_smem = std::max(smem, (size_t)116 * 1024);
      if (e->chr_slab) {
        static const int chain_ctas = getenv("BPPGPU_CHR_CHAIN_CTAS") ? atoi(getenv("BPPGPU_CHR_CHAIN_CTAS")) : 2;   // A/B knob
        if (chain_ctas >= 2) {
          q.nst = nst_level;
          chr_chain_slab_kernel<2><<<(unsigned)np, (kChrCons + 1) * 32, chr_slab_smem(S, nst_level), st>>>(q, e->chr_level_tile0[nlev] - q.tile0);
        } else {
          q.nst = nst_chain;
          chr_chain_slab_kernel<1><<<(unsigned)np, (kChrCons + 1) * 32, chr_slab_smem(S, nst_chain), st>>>(q, e->chr_level_tile0[nlev] - q.tile0);
        }
      } else {
        chr_chain_kernel<<<(unsigned)np, kChrWarps * 32, chain_smem, st>>>(q, e->chr_level_tile0[nlev] - q.tile0);
      }
      e->stats.kernel_launches++;
    }
    ChrRootParams rp{};
    rp.S = S; rp.nn = nn; rp.root = e->root; rp.p0 = f0;
    rp.flags = (e->flags & BPPGPU_FLAG_WEIGHTED_ROOT) ? 2u : 0u;
    rp.child_off = e->d_child_off; rp.children = e->d_children;
    rp.term = e->d_chr_term; rp.term_exp = e->d_chr_term_exp;
    rp.skip = e->d_chr_bad;
    rp.rootfreq_in = e->d_rootfreq; rp.rootfreq_used = e->d_rootfreq_used;
    rp.weights = e->d_weights; rp.site_lnl = e->d_site_lnl; rp.out = e->d_out; rp.out_stride = 1 + 2 * nn;
    chr_root_kernel<<<np, 256, S * sizeof(double), st>>>(rp);
    e->stats.kernel_launches++;
  }
  BPP_CUDA(cudaGetLastError());
  BPP_CUDA(cudaEventRecord(e->ring_b[e->ring_head], st));
  e->ring_head = (e->ring_head + 1) % bppgpu_engine::kRing;
  e->ring_n = std::min(e->ring_n + 1, (int)bppgpu_engine::kRing);
  // ---- the points for the table route, as ONE compact range [0, nbad) over gathered copies of their inputs ---------------------
  ranges.clear();
  std::vector<int> bad_idx;
  for (int p = 0; p < npts; ++p)
    if (e->chr_bad[p]) bad_idx.push_back(p);
  e->chr_table_points = (long long)bad_idx.size();
  e->chr_factored_points = npts - e->chr_table_points;
  e->stats.factored_points = e->chr_factored_points;
  e->stats.table_points = e->chr_table_points;
  if (!bad_idx.empty()) {
    const int nb = (int)bad_idx.size();
    if (nb > e->nbad_cap) {
      BPP_CUDA(cudaStreamSynchronize(st));
      for (void* q : {(void*)e->d_bad_idx, (void*)e->d_bad_brlen, (void*)e->d_bad_rootfreq, (void*)e->d_bad_rootfreq_used, (void*)e->d_bad_site_lnl,
                      (void*)e->d_bad_out, (void*)e->d_bad_branch_model})
        cudaFree(q);
      e->nbad_cap = std::min(npts, std::max(nb, 2 * e->nbad_cap));
      const size_t c = (size_t)e->nbad_cap;
      BPP_CUDA(dev_alloc(e, &e->d_bad_idx, c));
      BPP_CUDA(dev_alloc(e, &e->d_bad_brlen, c * nn));
      BPP_CUDA(dev_alloc(e, &e->d_bad_branch_model, c * nn));
      BPP_CUDA(dev_alloc(e, &e->d_bad_rootfreq, c * S));
      BPP_CUDA(dev_alloc(e, &e->d_bad_rootfreq_used, c * S));
      BPP_CUDA(dev_alloc(e, &e->d_bad_site_lnl, c * std::max<long long>(1, e->N)));
      BPP_CUDA(dev_alloc(e, &e->d_bad_out, c * (1 + 2 * nn)));
    }
    BPP_CUDA(cudaMemcpyAsync(e->d_bad_idx, bad_idx.data(), nb * sizeof(int), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaStreamSynchronize(st));   // bad_idx goes out of scope
    gather_rows_kernel<double><<<nb, 128, 0, st>>>(e->d_brlen, e->d_bad_brlen, e->d_bad_idx, nn);
    gather_rows_kernel<int><<<nb, 128, 0, st>>>(e->d_branch_model, e->d_bad_branch_model, e->d_bad_idx, nn);
    gather_rows_kernel<double><<<nb, 128, 0, st>>>(e->d_rootfreq, e->d_bad_rootfreq, e->d_bad_idx, S);
    gather_rows_kernel<double><<<nb, 128, 0, st>>>(e->d_rootfreq, e->d_bad_rootfreq_used, e->d_bad_idx, S);
    e->stats.kernel_launches += 4;
    ranges.push_back({0, nb});
  }
  e->stats.clv_updates += e->chr_factored_points * e->ni * (long long)S;
  (void)SS;
  return BPPGPU_OK;
}

static int eval_impl(bppgpu_engine* e, unsigned want, cudaStream_t st, bool timed, double* dev_out = nullptr) {
  e->last_point = -1;   // nothing is resident until this evaluation has been enqueued completely
  e->last_want = 0;
  int rc = check_ready(e);
  if (rc) return rc;
  if (want == 0) want = BPPGPU_EVAL_LNL;
  if (want & BPPGPU_EVAL_D2) want |= BPPGPU_EVAL_D1;
  const bool derivs = (want & (BPPGPU_EVAL_D1 | BPPGPU_EVAL_D2)) != 0;
  if (derivs && !e->keep) BPP_FAIL(BPPGPU_E_STATE, "derivatives need an engine created with BPPGPU_FLAG_KEEP_CLVS");
  if (derivs && e->path == PATH_POINTS)
    BPP_FAIL(BPPGPU_E_INVALID, "branch derivatives are not available on the batched-points path (n_points > 1)");
  // an evaluation enqueued on another stream (bppgpu_eval_device) must have finished with the engine's buffers
  if (e->eval_done && e->last_stream && e->last_stream != st) BPP_CUDA(cudaStreamWaitEvent(st, e->eval_done, 0));
  e->status_armed = false;
  rc = ensure_deriv_buffers(e, want);
  if (rc) return rc;
  bool any_series = false, any_chrd = false, any_real = false, any_complex = false;
  if (e->models_dirty) {
    std::vector<ModelDev> md(e->nmodels);
    for (int m = 0; m < e->nmodels; ++m) md[m] = to_dev(e->models[m]);
    BPP_CUDA(cudaMemcpyAsync(e->d_models, md.data(), md.size() * sizeof(ModelDev), cudaMemcpyHostToDevice, st));
    BPP_CUDA(cudaStreamSynchronize(st));
    e->models_dirty = false;
  }
  if (e->brlen_dirty_hi > e->brlen_dirty_lo) {
    const size_t off = (size_t)e->brlen_dirty_lo * e->nn, cnt = (size_t)(e->brlen_dirty_hi - e->brlen_dirty_lo) * e->nn;
    BPP_CUDA(cudaMemcpyAsync(e->d_brlen + off, e->h_brlen.data() + off, cnt * 8, cudaMemcpyHostToDevice, st));   // (pageable source: staged before the call returns)
    e->brlen_dirty_lo = e->brlen_dirty_hi = 0;
  }
  for (int m = 0; m < e->nmodels; ++m) {
    if (!e->models[m].set) continue;
    if (!(e->models[m].flags & BPPGPU_MODEL_NONSINGULAR)) any_series = true;
    else {
      if (e->models[m].flags & BPPGPU_MODEL_CHR_DERIV) any_chrd = true;
      if (e->models[m].has_complex) any_complex = true;
      else any_real = true;
    }
  }
  rc = ensure_scratch(e, any_series, any_chrd && derivs);
  if (rc) return rc;
  if (any_series || any_chrd) {   // only the series / Chromosome kernels ever raise the status word
    BPP_CUDA(cudaMemsetAsync(e->d_status, 0, sizeof(int), st));
    e->status_armed = true;
  }
  e->stats.kernel_launches = 0;
  e->stats.clv_updates = 0;
  const int S = e->S, C = e->C, nn = e->nn;
  const size_t SS = (size_t)S * S;
  unsigned pt_want = BPPGPU_WANT_P | ((want & BPPGPU_EVAL_D1) ? BPPGPU_WANT_DP : 0) | ((want & BPPGPU_EVAL_D2) ? BPPGPU_WANT_D2P : 0);
  if (timed) BPP_CUDA(cudaEventRecord(e->ev0, st));
  if (e->rootfreq_used_stale || (e->flags & BPPGPU_FLAG_WEIGHTED_ROOT)) {   // the copy in use differs from the input only with weighted roots
    BPP_CUDA(cudaMemcpyAsync(e->d_rootfreq_used, e->d_rootfreq, (size_t)e->npoints * S * 8, cudaMemcpyDeviceToDevice, st));
    e->rootfreq_used_stale = false;
  }
  std::vector<std::pair<int, int>> ranges(1, {0, e->npoints});
  if (e->chr_factored) {
    rc = eval_points_factored(e, st, any_real, any_complex, ranges);
    if (rc) return rc;
    if (!ranges.empty()) {
      rc = ensure_tables(e);
      if (rc) return rc;
      rc = ensure_scratch(e, any_series, false);
      if (rc) return rc;
    }
    e->last_point = e->npoints - 1;
  }
  // per-point arrays the table route reads and writes: the engine's own, or the compact copies of a factored engine
  const bool compact = e->chr_factored;
  const int* pa_bm = compact ? e->d_bad_branch_model : e->d_branch_model;
  const double* pa_brlen = compact ? e->d_bad_brlen : e->d_brlen;
  const double* pa_rootfreq = compact ? e->d_bad_rootfreq : e->d_rootfreq;
  double* pa_rootfreq_used = compact ? e->d_bad_rootfreq_used : e->d_rootfreq_used;
  double* pa_site_lnl = compact ? e->d_bad_site_lnl : e->d_site_lnl;
  double* pa_out = compact ? e->d_bad_out : e->d_out;
  for (const auto& range : ranges)
  for (int p0 = range.first; p0 < range.second; p0 += e->pchunk) {
    const int np = std::min(e->pchunk, range.second - p0);
    const bool first_chunk = p0 == ranges.front().first, last_chunk = p0 + np >= ranges.back().second;
    long long launches = 0;
    // DNA walk, real spectra, plain models: P(t) is built inside the stream-packing launch (pt_pack4c_kernel)
    bool clamp_or_chr = false;
    for (int m = 0; m < e->nmodels; ++m)
      if (e->models[m].set && (e->models[m].flags & (BPPGPU_MODEL_CLAMP01 | BPPGPU_MODEL_CHR_DERIV))) clamp_or_chr = true;
    const bool fused_pt = e->w4c && S == 4 && !any_series && !any_complex && !clamp_or_chr && pt_want == BPPGPU_WANT_P;
    BPP_CUDA(cudaEventRecord(e->ptring_a[e->ptring_head], st));
    if (!fused_pt)
    rc = launch_pt(st, e->d_models, any_series, any_chrd, any_real, any_complex, e->homogeneous_points, pa_bm + (size_t)p0 * nn,
                   pa_brlen + (size_t)p0 * nn, e->d_rates, S, C, nn, e->root, np, pt_want, e->d_P, e->d_dP, e->d_d2P,
                   e->d_scratch, e->d_status, &launches);
    if (rc) return rc;
    BPP_CUDA(cudaEventRecord(e->ptring_b[e->ptring_head], st));
    e->ptring_head = (e->ptring_head + 1) % bppgpu_engine::kRing;
    e->ptring_n = std::min(e->ptring_n + 1, (int)bppgpu_engine::kRing);
    e->stats.kernel_launches += launches;
    if (e->w4c) {
      if (e->codesT_dirty && e->N > 0) {
        for (const auto& sg : e->w4c_segs) {
          pack_codesC_kernel<<<(unsigned)sg.grid, 256, 0, st>>>(
              (const unsigned char*)e->d_codes, e->d_w4c_tip_order, (int)e->w4c_tip_order.size(), e->ncodes, e->N, sg.pat0, sg.pat_end,
              (e->w4c_nw / C) * 32 * sg.pt, e->d_codesC + sg.codes_off);
          e->stats.kernel_launches++;
        }
        e->codesT_dirty = false;
      }
      for (int pl = 0; pl < np; ++pl) {
        if (fused_pt) {
          PtPack4cParams pk{};
          pk.blocks = e->d_w4c_blocks; pk.models = e->d_models;
          pk.branch_model = pa_bm + (size_t)(p0 + pl) * nn;
          pk.brlen = pa_brlen + (size_t)(p0 + pl) * nn;
          pk.rates = e->d_rates; pk.code_table = e->d_code_table; pk.C = C; pk.ncodes = e->ncodes;
          pk.P = e->d_P + (size_t)pl * nn * C * SS;
          pk.stream = e->d_w4c_stream + (size_t)pl * e->w4c_stream_bytes;
          pt_pack4c_kernel<<<(unsigned)e->w4c_blocks.size(), 64, 0, st>>>(pk);
        } else {
          pack_stream4c_kernel<<<(unsigned)e->w4c_blocks.size(), 64, 0, st>>>(
              e->d_w4c_blocks, e->d_P + (size_t)pl * nn * C * SS, e->d_code_table, C, e->ncodes,
              e->d_w4c_stream + (size_t)pl * e->w4c_stream_bytes);
        }
      }
      e->stats.kernel_launches += np;
    } else if (e->path == PATH_WALK4) {
      if (e->codesT_dirty && e->N > 0) {
        transpose_codes_kernel<<<(unsigned)((e->N + 127) / 128), 128, 0, st>>>(
            (const unsigned char*)e->d_codes, e->d_w4_tip_order, (int)e->w4_tip_order.size(), e->N, e->w4_tstride, e->d_codesT);
        e->stats.kernel_launches++;
        e->codesT_dirty = false;
      }
      for (int pl = 0; pl < np; ++pl)
        pack_stream4_kernel<<<(unsigned)e->w4_blocks.size(), 64, 0, st>>>(
            e->d_w4_blocks, e->d_P + (size_t)pl * nn * C * SS, e->d_code_table, C, e->ncodes,
            e->d_w4_stream + (size_t)pl * e->w4_stream_len);
      e->stats.kernel_launches += np;
    }
    if (e->d_tiptab) {
      TipTabParams tp{};
      tp.P = e->d_P;
      tp.code_table = e->d_code_table;
      tp.leaf_nodes = e->d_leaf_nodes;
      tp.S = S; tp.C = C; tp.nn = nn; tp.nl = e->nl; tp.ncodes = e->ncodes;
      tp.tiptab = e->d_tiptab;
      tiptab_kernel<<<np * e->nl * C, 128, 0, st>>>(tp);
      e->stats.kernel_launches++;
      if (e->path == PATH_DMMA && derivs) {
        tp.P = e->d_dP; tp.tiptab = e->d_dtiptab;
        tiptab_kernel<<<np * e->nl * C, 128, 0, st>>>(tp);
        e->stats.kernel_launches++;
        if (want & BPPGPU_EVAL_D2) {
          tp.P = e->d_d2P; tp.tiptab = e->d_d2tiptab;
          tiptab_kernel<<<np * e->nl * C, 128, 0, st>>>(tp);
          e->stats.kernel_launches++;
        }
      }
    }
    if (e->prune64) {
      prune_pack_kernel<64><<<nn * C, 256, 0, st>>>(e->d_P, e->d_fam_packL);
      e->stats.kernel_launches++;
    }
    if (e->family) {
      // operands in fragment order for the S = 20 tensor-core kernels (single-point engines only)
      FamilyPackParams pk{};
      pk.P = e->d_P;
      pk.dP = derivs ? e->d_dP : nullptr;
      pk.d2P = (want & BPPGPU_EVAL_D2) ? e->d_d2P : nullptr;
      pk.packA = e->d_fam_packA; pk.packS = e->d_fam_packS; pk.packL = e->d_fam_packL;
      pk.S = S;
      pk.nbc = nn * C;
      pk.ntc = derivs ? e->nl * C * e->ncodes : 0;
      if (derivs) {
        pk.tt = e->d_tiptab;
        pk.dtt = e->d_dtiptab;
        pk.d2tt = (want & BPPGPU_EVAL_D2) ? e->d_d2tiptab : nullptr;
        pk.packT = e->d_fam_packT;
      }
      family_pack_kernel<<<pk.nbc + (pk.ntc + 3) / 4, 256, 0, st>>>(pk);
      e->stats.kernel_launches++;
    }
    BPP_CUDA(cudaGetLastError());
    if (e->path == PATH_POINTS) {
      if (first_chunk) BPP_CUDA(cudaEventRecord(e->ring_a[e->ring_head], st));
      const long long rows = e->N * C;
      for (const Op& op : e->gprog.ops) {
        PointsNodeParams pp{};
        pp.childs = e->gprog.d_childs + op.child_begin;
        pp.nchild = op.nchild;
        pp.out_idx = op.keep_idx;
        pp.S = S; pp.C = C; pp.nn = nn; pp.nl = e->nl; pp.ni = e->ni; pp.ncodes = e->ncodes; pp.code_bytes = e->code_bytes;
        pp.N = e->N;
        pp.P = e->d_P; pp.code_table = e->d_code_table; pp.code_single = e->d_code_single; pp.codes = e->d_codes;
        pp.keep = e->d_keep; pp.keep_exp = e->d_keep_exp;
        // a chunk holds only a few hundred points (one CTA each per row): large alphabets get 16 warps per CTA so that enough
        // of the point's P rows are in flight to stream them at HBM speed
        static const int pts_threads_env = getenv("BPPGPU_POINTS_THREADS") ? atoi(getenv("BPPGPU_POINTS_THREADS")) : 0;
        const int pts_threads = pts_threads_env > 0 ? pts_threads_env : (S >= 128 ? 512 : 256);  // S = 200, 256 points: 27.0 ms (256 threads), 16.7 (512), 19.4 (1024)
        points_node_kernel<<<dim3((unsigned)np, (unsigned)std::min<long long>(rows, 64)), pts_threads, (2 * S + 32) * sizeof(double), st>>>(pp);
        e->stats.kernel_launches++;
      }
      PointsRootParams pr{};
      pr.root_idx = e->internal_idx[e->root]; pr.S = S; pr.C = C; pr.ni = e->ni;
      pr.flags = ((e->flags & BPPGPU_FLAG_R_SEMANTICS) ? 1u : 0u) | ((e->flags & BPPGPU_FLAG_WEIGHTED_ROOT) ? 2u : 0u);
      pr.N = e->N;
      pr.keep = e->d_keep; pr.keep_exp = e->d_keep_exp; pr.probs = e->d_probs; pr.weights = e->d_weights;
      pr.rootfreq_in = pa_rootfreq + (size_t)p0 * S;
      pr.rootfreq_used = pa_rootfreq_used + (size_t)p0 * S;
      pr.site_lnl = pa_site_lnl + (size_t)p0 * e->N;
      pr.out = pa_out + (size_t)p0 * (1 + 2 * nn);
      pr.out_stride = 1 + 2 * nn;
      points_root_kernel<<<np, 256, S * sizeof(double), st>>>(pr);
      e->stats.kernel_launches++;
      BPP_CUDA(cudaGetLastError());
      e->stats.clv_updates += (long long)np * e->ni * rows * S;
      if (last_chunk) {
        BPP_CUDA(cudaEventRecord(e->ring_b[e->ring_head], st));
        e->ring_head = (e->ring_head + 1) % bppgpu_engine::kRing;
        e->ring_n = std::min(e->ring_n + 1, (int)bppgpu_engine::kRing);
      }
      e->last_point = p0 + np - 1;
      continue;
    }
    for (int pl = 0; pl < np; ++pl) {
      const int point = p0 + pl;
      if (point == 0) BPP_CUDA(cudaEventRecord(e->ring_a[e->ring_head], st));
      rc = enqueue_prune(e, point, pl, st);
      if (rc) return rc;
      if (point == 0) {
        BPP_CUDA(cudaEventRecord(e->ring_b[e->ring_head], st));
        e->ring_head = (e->ring_head + 1) % bppgpu_engine::kRing;
        e->ring_n = std::min(e->ring_n + 1, (int)bppgpu_engine::kRing);
      }
      if (derivs) {
        rc = enqueue_derivs(e, point, pl, want, st);
        if (rc) return rc;
      }
      e->last_point = point;
    }
  }
  (void)SS;
  if (compact && !ranges.empty()) {   // results of the table-route points back to their places
    const int nb = ranges.front().second;
    scatter_rows_kernel<double><<<nb, 128, 0, st>>>(e->d_bad_out, e->d_out, e->d_bad_idx, 1 + 2 * nn, 1);
    scatter_rows_kernel<double><<<nb, 128, 0, st>>>(e->d_bad_site_lnl, e->d_site_lnl, e->d_bad_idx, (int)e->N, (int)e->N);
    scatter_rows_kernel<double><<<nb, 128, 0, st>>>(e->d_bad_rootfreq_used, e->d_rootfreq_used, e->d_bad_idx, S, S);
    e->stats.kernel_launches += 3;
    BPP_CUDA(cudaGetLastError());
  }
  const size_t row = (size_t)(1 + 2 * nn);
  // what the caller can read: one point and no derivatives -> the first element only (an 8-byte message, not 16 nn + 8 bytes)
  const size_t live = (e->npoints == 1 && !derivs) ? 1 : (size_t)e->npoints * row;
  if (e->comm && e->comm_nranks > 1) {   // pattern shards: every rank ends up with the whole alignment's lnL, d1, d2 -- straight
    BPP_NCCL(nccl_api().AllReduce(e->d_out, dev_out ? dev_out : e->d_out, live, ncclDouble, ncclSum, (ncclComm_t)e->comm, st));   // into the caller's buffer
  } else if (dev_out) {
    BPP_CUDA(cudaMemcpyAsync(dev_out, e->d_out, live * 8, cudaMemcpyDeviceToDevice, st));
  }
  if (timed) BPP_CUDA(cudaEventRecord(e->ev1, st));
  BPP_CUDA(cudaEventRecord(e->eval_done, st));
  e->last_stream = st;
  e->last_want = want;
  return BPPGPU_OK;
}

int bppgpu_eval(bppgpu_engine* e, unsigned want, double* lnl, double* d1, double* d2) {
  ENGINE_ENTER(e);
  int rc = eval_impl(e, want, e->stream, true);
  if (rc) return rc;
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  float ms = 0.f;
  BPP_CUDA(cudaEventElapsedTime(&ms, e->ev0, e->ev1));
  e->stats.last_eval_ms = ms;
  {
    const int last = (e->ring_head + bppgpu_engine::kRing - 1) % bppgpu_engine::kRing;
    if (e->ring_n > 0 && cudaEventElapsedTime(&ms, e->ring_a[last], e->ring_b[last]) == cudaSuccess) e->stats.prune_ms = ms;
  }
  const int nn = e->nn;
  std::vector<double> h((size_t)e->npoints * (1 + 2 * nn));
  BPP_CUDA(cudaMemcpy(h.data(), e->d_out, h.size() * 8, cudaMemcpyDeviceToHost));
  int status = 0;
  if (e->status_armed) BPP_CUDA(cudaMemcpy(&status, e->d_status, 4, cudaMemcpyDeviceToHost));
  if (status) BPP_FAIL(BPPGPU_E_NUMERIC, "ChromosomeSubstitutionModel: Taylor series did not reach convergence!");
  for (int p = 0; p < e->npoints; ++p) {
    const double* row = h.data() + (size_t)p * (1 + 2 * nn);
    if (lnl) lnl[p] = row[0];
    if (d1 && (e->last_want & BPPGPU_EVAL_D1)) std::copy(row + 1, row + 1 + nn, d1 + (size_t)p * nn);
    if (d2 && (e->last_want & BPPGPU_EVAL_D2)) std::copy(row + 1 + nn, row + 1 + 2 * nn, d2 + (size_t)p * nn);
  }
  return BPPGPU_OK;
}

int bppgpu_eval_device(bppgpu_engine* e, unsigned want, double* dev_out, void* cuda_stream) {
  ENGINE_ENTER(e);
  if (!dev_out) BPP_FAIL(BPPGPU_E_INVALID, "null dev_out");
  cudaStream_t st = cuda_stream ? (cudaStream_t)cuda_stream : e->stream;
  return eval_impl(e, want, st, false, dev_out);
}

// ---- accessors -------------------------------------------------------------------------
int bppgpu_get_site_lnl(bppgpu_engine* e, int32_t point, double* out) {
  ENGINE_SYNC(e);
  if (point < 0 || point >= e->npoints || !out) BPP_FAIL(BPPGPU_E_INVALID, "bad point or null out");
  if (e->last_want == 0) BPP_FAIL(BPPGPU_E_STATE, "no evaluation yet");
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  BPP_CUDA(cudaMemcpy(out, e->d_site_lnl + (size_t)point * e->N, (size_t)e->N * 8, cudaMemcpyDeviceToHost));
  return BPPGPU_OK;
}

// class-major device slabs -> the reference's VVVdouble order [pattern][class][state] (host side, accessor only)
static void to_reference_order(bppgpu_engine* e, double* clv, int32_t* ex) {
  if (!e->clv_class_major || e->C == 1) return;
  const size_t N = (size_t)e->N, C = (size_t)e->C, S = (size_t)e->S;
  std::vector<double> t(clv, clv + N * C * S);
  for (size_t c = 0; c < C; ++c)
    for (size_t i = 0; i < N; ++i) memcpy(clv + (i * C + c) * S, t.data() + (c * N + i) * S, S * sizeof(double));
  if (ex) {
    std::vector<int32_t> te(ex, ex + N * C);
    for (size_t c = 0; c < C; ++c)
      for (size_t i = 0; i < N; ++i) ex[i * C + c] = te[c * N + i];
  }
}

int bppgpu_get_clv(bppgpu_engine* e, int32_t point, int32_t node, int32_t which, double* clv, int32_t* scale_exp) {
  ENGINE_SYNC(e);
  if (!e->keep) BPP_FAIL(BPPGPU_E_STATE, "bppgpu_get_clv needs BPPGPU_FLAG_KEEP_CLVS");
  if (node < 0 || node >= e->nn || !clv || point < 0 || point >= e->npoints) BPP_FAIL(BPPGPU_E_INVALID, "bad node / point or null out");
  const size_t clvn = (size_t)e->N * e->C * e->S;
  size_t pt_off = 0;  // slab offset of the point inside the resident chunk (batched-points path)
  if (e->chr_factored) BPP_FAIL(BPPGPU_E_STATE, "the factored batched-points route keeps no per-node arrays: create the engine with BPPGPU_FLAG_KEEP_CLVS");
  if (e->path == PATH_POINTS) {
    const int chunk0 = ((e->npoints - 1) / e->pchunk) * e->pchunk;
    if (e->last_point < 0 || point < chunk0 || point >= e->npoints)
      BPP_FAIL(BPPGPU_E_STATE, "CLVs resident are those of points >= %d", chunk0);
    pt_off = (size_t)(point - chunk0) * e->ni;
  } else if (point != e->last_point) {
    BPP_FAIL(BPPGPU_E_STATE, "CLVs resident are those of point %d", e->last_point);
  }
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  if (which == 0) {
    if (e->internal_idx[node] < 0) BPP_FAIL(BPPGPU_E_INVALID, "node %d is a leaf: its CLV is the code table row", node);
    const size_t k = pt_off + (size_t)e->internal_idx[node];
    BPP_CUDA(cudaMemcpy(clv, e->d_keep + k * clvn, clvn * 8, cudaMemcpyDeviceToHost));
    if (scale_exp) BPP_CUDA(cudaMemcpy(scale_exp, e->d_keep_exp + k * e->N * e->C, (size_t)e->N * e->C * 4, cudaMemcpyDeviceToHost));
    to_reference_order(e, clv, scale_exp);
  } else {
    if (!(e->last_want & BPPGPU_EVAL_D1) || !e->d_upper) BPP_FAIL(BPPGPU_E_STATE, "upper CLVs exist after an eval with derivatives");
    if (node == e->root) BPP_FAIL(BPPGPU_E_INVALID, "the root has no upper CLV");
    const int slab = e->upper_slab[node];
    if (slab < 0) BPP_FAIL(BPPGPU_E_STATE, "the upper CLV of tip %d is not materialised at this problem size", node);
    BPP_CUDA(cudaMemcpy(clv, e->d_upper + (size_t)slab * clvn, clvn * 8, cudaMemcpyDeviceToHost));
    if (scale_exp) BPP_CUDA(cudaMemcpy(scale_exp, e->d_upper_exp + (size_t)slab * e->N * e->C, (size_t)e->N * e->C * 4, cudaMemcpyDeviceToHost));
    to_reference_order(e, clv, scale_exp);
  }
  return BPPGPU_OK;
}

int bppgpu_get_node_posteriors(bppgpu_engine* e, int32_t point, int32_t node, double* full_out, int32_t* exp_out, double* post_out) {
  ENGINE_SYNC(e);
  if (!e->keep) BPP_FAIL(BPPGPU_E_STATE, "bppgpu_get_node_posteriors needs BPPGPU_FLAG_KEEP_CLVS");
  if (node < 0 || node >= e->nn || point < 0 || point >= e->npoints) BPP_FAIL(BPPGPU_E_INVALID, "bad node or point");
  if (e->path == PATH_POINTS) BPP_FAIL(BPPGPU_E_STATE, "not available on the batched-points path");
  if (point != e->last_point) BPP_FAIL(BPPGPU_E_STATE, "CLVs resident are those of point %d", e->last_point);
  const bool leaf = e->leaf_slot[node] >= 0, root = node == e->root;
  const int S = e->S, C = e->C;
  const long long N = e->N;
  if (N == 0) return BPPGPU_OK;
  const size_t clvn = (size_t)N * C * S, rows = (size_t)N * C;
  const bool need_full = full_out || exp_out || (post_out && !leaf);
  const int uslab = root ? -1 : (e->d_upper ? e->upper_slab[node] : -1);
  if (need_full && !root) {
    if (!(e->last_want & BPPGPU_EVAL_D1) || !e->d_upper) BPP_FAIL(BPPGPU_E_STATE, "upper CLVs exist after an eval with derivatives");
    if (uslab < 0) BPP_FAIL(BPPGPU_E_STATE, "the upper CLV of tip %d is not materialised at this problem size", node);
  }
  cudaStream_t st = e->stream;
  double *d_full = nullptr, *d_post = nullptr;
  int* d_fexp = nullptr;
  auto cleanup = [&]() { cudaFree(d_full); cudaFree(d_post); cudaFree(d_fexp); };
  if (need_full) {
    if (cudaMalloc(&d_full, clvn * 8) != cudaSuccess || cudaMalloc(&d_fexp, rows * 4) != cudaSuccess) {
      cleanup();
      BPP_FAIL(BPPGPU_E_NOMEM, "out of device memory for the likelihood array of node %d", node);
    }
    NodeFullParams np{};
    np.is_leaf = leaf; np.is_root = root;
    np.S = S; np.C = C; np.code_bytes = e->code_bytes; np.N = N;
    np.prow = e->clv_class_major ? 1 : C;
    np.crow = e->clv_class_major ? N : 1;
    const int pl = e->path == PATH_POINTS ? 0 : (point % e->pchunk);
    np.P = e->d_P + ((size_t)pl * e->nn + node) * C * S * S;
    if (leaf) {
      np.codes = (const char*)e->d_codes + (size_t)e->leaf_slot[node] * N * e->code_bytes;
      np.code_table = e->d_code_table;
    } else {
      np.lower = e->d_keep + (size_t)e->internal_idx[node] * clvn;
      np.lower_exp = e->d_keep_exp + (size_t)e->internal_idx[node] * rows;
    }
    if (!root) {
      np.upper = e->d_upper + (size_t)uslab * clvn;
      np.upper_exp = e->d_upper_exp + (size_t)uslab * rows;
    }
    np.rootfreq = e->d_rootfreq_used + (size_t)point * S;
    np.out = d_full; np.out_exp = d_fexp;
    const int grid = (int)std::min<long long>(((long long)clvn + 255) / 256, (long long)g_sm_count * 32);
    node_full_kernel<<<grid, 256, 0, st>>>(np);
  }
  if (post_out) {
    if (cudaMalloc(&d_post, clvn * 8) != cudaSuccess) {
      cleanup();
      BPP_FAIL(BPPGPU_E_NOMEM, "out of device memory for the posteriors of node %d", node);
    }
    const void* codes = leaf ? (const void*)((const char*)e->d_codes + (size_t)e->leaf_slot[node] * N * e->code_bytes) : nullptr;
    node_posterior_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(d_full, d_fexp, leaf ? 1 : 0, codes, e->code_bytes,
                                                                       e->d_code_table, e->d_probs, S, C, N, d_post);
  }
  cudaError_t err = cudaGetLastError();
  if (err == cudaSuccess && full_out) err = cudaMemcpyAsync(full_out, d_full, clvn * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess && exp_out) err = cudaMemcpyAsync(exp_out, d_fexp, rows * 4, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess && post_out) err = cudaMemcpyAsync(post_out, d_post, clvn * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess) err = cudaStreamSynchronize(st);
  cleanup();
  BPP_CUDA(err);
  return BPPGPU_OK;
}

int bppgpu_get_marginal_posteriors(bppgpu_engine* e, int32_t point, int32_t node, double* post_out, double* joint_out) {
  ENGINE_SYNC(e);
  if (!e->keep) BPP_FAIL(BPPGPU_E_STATE, "bppgpu_get_marginal_posteriors needs BPPGPU_FLAG_KEEP_CLVS");
  if (node < 0 || node >= e->nn || !post_out || point < 0 || point >= e->npoints) BPP_FAIL(BPPGPU_E_INVALID, "bad node / point or null out");
  if (e->path == PATH_POINTS) BPP_FAIL(BPPGPU_E_STATE, "not available on the batched-points path");
  if (e->last_want == 0) BPP_FAIL(BPPGPU_E_STATE, "no evaluation yet");
  if (point != e->last_point) BPP_FAIL(BPPGPU_E_STATE, "CLVs resident are those of point %d", e->last_point);
  const bool leaf = e->leaf_slot[node] >= 0, root = node == e->root;
  if (root && joint_out) BPP_FAIL(BPPGPU_E_INVALID, "the root has no father: no joint posterior");
  const int S = e->S, C = e->C;
  const long long N = e->N;
  if (N == 0) return BPPGPU_OK;
  const size_t clvn = (size_t)N * C * S, rows = (size_t)N * C;
  int uslab = -1;
  if (!root) {
    if (!(e->last_want & BPPGPU_EVAL_D1) || !e->d_upper) BPP_FAIL(BPPGPU_E_STATE, "upper CLVs exist after an eval with derivatives");
    uslab = e->upper_slab[node];
    if (uslab < 0) BPP_FAIL(BPPGPU_E_STATE, "the upper CLV of tip %d is not materialised at this problem size", node);
  }
  double *d_post = nullptr, *d_joint = nullptr;
  auto cleanup = [&]() { cudaFree(d_post); cudaFree(d_joint); };
  if (cudaMalloc(&d_post, (size_t)N * S * 8) != cudaSuccess ||
      (joint_out && cudaMalloc(&d_joint, (size_t)N * S * S * 8) != cudaSuccess)) {
    cleanup();
    cudaGetLastError();
    BPP_FAIL(BPPGPU_E_NOMEM, "out of device memory for the marginal posteriors of node %d", node);
  }
  MarginalParams mp{};
  mp.is_leaf = leaf; mp.is_root = root;
  mp.S = S; mp.C = C; mp.code_bytes = e->code_bytes; mp.N = N;
  mp.prow = e->clv_class_major ? 1 : C;
  mp.crow = e->clv_class_major ? N : 1;
  mp.P = e->d_P + ((size_t)(point % e->pchunk) * e->nn + node) * C * S * S;
  if (leaf) {
    mp.codes = (const char*)e->d_codes + (size_t)e->leaf_slot[node] * N * e->code_bytes;
    mp.code_table = e->d_code_table;
  } else {
    mp.lower = e->d_keep + (size_t)e->internal_idx[node] * clvn;
    mp.lower_exp = e->d_keep_exp + (size_t)e->internal_idx[node] * rows;
  }
  if (!root) {
    mp.upper = e->d_upper + (size_t)uslab * clvn;
    mp.upper_exp = e->d_upper_exp + (size_t)uslab * rows;
  }
  mp.rootfreq = e->d_rootfreq_used + (size_t)point * S;
  mp.probs = e->d_probs; mp.SR = e->d_SR; mp.rexp = e->d_rexp;
  mp.post = d_post; mp.joint = d_joint;
  cudaStream_t st = e->stream;
  const int grid = (int)std::min<long long>((N * S + 127) / 128, (long long)g_sm_count * 32);
  marginal_posterior_kernel<<<grid, 128, 0, st>>>(mp);
  cudaError_t err = cudaGetLastError();
  if (err == cudaSuccess) err = cudaMemcpyAsync(post_out, d_post, (size_t)N * S * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess && joint_out) err = cudaMemcpyAsync(joint_out, d_joint, (size_t)N * S * S * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess) err = cudaStreamSynchronize(st);
  cleanup();
  BPP_CUDA(err);
  return BPPGPU_OK;
}

int bppgpu_ml_ancestral_states(bppgpu_engine* e, int32_t point, int32_t* states, double* best_lnl) {
  ENGINE_SYNC(e);
  if (!states || point < 0 || point >= e->npoints) BPP_FAIL(BPPGPU_E_INVALID, "null states or bad point");
  if (e->path == PATH_POINTS) BPP_FAIL(BPPGPU_E_STATE, "not available on the batched-points path");
  if (e->last_want == 0) BPP_FAIL(BPPGPU_E_STATE, "no evaluation yet (the transition probabilities of the last evaluation are used)");
  if (point != e->last_point) BPP_FAIL(BPPGPU_E_STATE, "tables resident are those of point %d", e->last_point);
  const int S = e->S, C = e->C, nn = e->nn;
  const long long N = e->N;
  if ((size_t)4 * S * sizeof(double) > 48 * 1024) BPP_FAIL(BPPGPU_E_INVALID, "joint ML reconstruction supports up to 1536 states (%d given)", S);
  for (int n = 0; n < nn; ++n)
    if (e->child_off[n + 1] - e->child_off[n] > 4) BPP_FAIL(BPPGPU_E_INVALID, "node %d has more than 4 sons", n);
  if (N == 0) return BPPGPU_OK;
  const size_t clvn = (size_t)N * C * S, rows = (size_t)N * C;
  // slabs: the arrays of a node live until its father is done; the traceback tables of every node stay
  std::vector<double*> L(nn, nullptr);
  std::vector<int*> E(nn, nullptr);
  std::vector<double*> freeL;
  std::vector<int*> freeE;
  unsigned short* d_anc = nullptr;
  int* d_state = nullptr;
  double* d_best = nullptr;
  auto cleanup = [&]() {
    for (double* q : L) cudaFree(q);
    for (int* q : E) cudaFree(q);
    for (double* q : freeL) cudaFree(q);
    for (int* q : freeE) cudaFree(q);
    cudaFree(d_anc); cudaFree(d_state); cudaFree(d_best);
    cudaGetLastError();
  };
#define ML_TRY(expr)                                                                         \
  do {                                                                                       \
    cudaError_t _r = (expr);                                                                 \
    if (_r != cudaSuccess) {                                                                 \
      cleanup();                                                                             \
      BPP_FAIL(_r == cudaErrorMemoryAllocation ? BPPGPU_E_NOMEM : BPPGPU_E_CUDA,            \
               "joint ML reconstruction: %s", cudaGetErrorString(_r));                       \
    }                                                                                        \
  } while (0)
  ML_TRY(cudaMalloc(&d_anc, (size_t)nn * N * S * sizeof(unsigned short)));
  ML_TRY(cudaMalloc(&d_state, (size_t)nn * N * sizeof(int)));
  if (best_lnl) ML_TRY(cudaMalloc(&d_best, (size_t)N * 8));
  cudaStream_t st = e->stream;
  const int pl = point % e->pchunk;
  const int wpb = 4;   // warps (rows) per block
  const unsigned grid = (unsigned)((rows + wpb - 1) / wpb);
  const size_t smem = (size_t)wpb * S * sizeof(double);
  for (int k = nn - 1; k >= 0; --k) {   // reverse pre-order: sons before fathers
    const int n = e->preorder[k];
    if (!freeL.empty()) { L[n] = freeL.back(); freeL.pop_back(); E[n] = freeE.back(); freeE.pop_back(); }
    else { ML_TRY(cudaMalloc(&L[n], clvn * 8)); ML_TRY(cudaMalloc(&E[n], rows * 4)); }
    MLNodeParams mp{};
    const bool leaf = e->leaf_slot[n] >= 0;
    mp.kind = leaf ? 0 : (n == e->root ? 2 : 1);
    mp.S = S; mp.C = C; mp.code_bytes = e->code_bytes; mp.N = N;
    mp.P = e->d_P + ((size_t)pl * nn + n) * C * S * S;
    mp.code_table = e->d_code_table;
    mp.rootfreq = e->d_rootfreq_used + (size_t)point * S;
    if (leaf) mp.codes = (const char*)e->d_codes + (size_t)e->leaf_slot[n] * N * e->code_bytes;
    mp.nson = e->child_off[n + 1] - e->child_off[n];
    for (int j = 0; j < mp.nson; ++j) {
      const int sn = e->children[e->child_off[n] + j];
      mp.son_L[j] = L[sn];
      mp.son_E[j] = E[sn];
    }
    mp.L = L[n]; mp.E = E[n];
    mp.anc = d_anc + (size_t)n * N * S;
    ml_node_kernel<<<grid, wpb * 32, smem, st>>>(mp);
    ML_TRY(cudaGetLastError());
    for (int j = 0; j < mp.nson; ++j) {   // stream order keeps the slab valid until the kernel above has read it
      const int sn = e->children[e->child_off[n] + j];
      freeL.push_back(L[sn]); freeE.push_back(E[sn]);
      L[sn] = nullptr; E[sn] = nullptr;
    }
  }
  const unsigned gridN = (unsigned)((N + 127) / 128);
  ml_root_state_kernel<<<gridN, 128, 0, st>>>(L[e->root], E[e->root], S, C, N, d_state + (size_t)e->root * N, d_best);
  for (int k = 0; k < nn; ++k) {   // fathers before sons
    const int n = e->preorder[k];
    if (n == e->root) continue;
    ml_traceback_kernel<<<gridN, 128, 0, st>>>(d_anc + (size_t)n * N * S, d_state + (size_t)e->parent[n] * N, S, N, d_state + (size_t)n * N);
  }
  ML_TRY(cudaGetLastError());
  ML_TRY(cudaMemcpyAsync(states, d_state, (size_t)nn * N * sizeof(int), cudaMemcpyDeviceToHost, st));
  if (best_lnl) ML_TRY(cudaMemcpyAsync(best_lnl, d_best, (size_t)N * 8, cudaMemcpyDeviceToHost, st));
  ML_TRY(cudaStreamSynchronize(st));
#undef ML_TRY
  cleanup();
  return BPPGPU_OK;
}

int bppgpu_get_root_reparam_derivatives(bppgpu_engine* e, int32_t point, double out[4]) {
  ENGINE_SYNC(e);
  if (!out || point < 0 || point >= e->npoints) BPP_FAIL(BPPGPU_E_INVALID, "null out or bad point");
  if (!e->keep) BPP_FAIL(BPPGPU_E_STATE, "bppgpu_get_root_reparam_derivatives needs BPPGPU_FLAG_KEEP_CLVS");
  if (e->path == PATH_POINTS) BPP_FAIL(BPPGPU_E_STATE, "not available on the batched-points path");
  if (point != e->last_point) BPP_FAIL(BPPGPU_E_STATE, "CLVs resident are those of point %d", e->last_point);
  if (!(e->last_want & BPPGPU_EVAL_D2) || !e->d_dP || !e->d_d2P)
    BPP_FAIL(BPPGPU_E_STATE, "BrLenRoot / RootPosition derivatives need an eval with BPPGPU_EVAL_D2");
  const int root = e->root;
  const int ns = e->child_off[root + 1] - e->child_off[root];
  if (ns < 2 || ns > 4) BPP_FAIL(BPPGPU_E_INVALID, "the root must have 2 to 4 sons (it has %d)", ns);
  const int S = e->S, C = e->C;
  const long long N = e->N;
  for (int k = 0; k < 4; ++k) out[k] = 0.0;
  if (N == 0) return BPPGPU_OK;
  const size_t clvn = (size_t)N * C * S, rows = (size_t)N * C, SS = (size_t)S * S;
  const int pl = point % e->pchunk;
  RootReparamParams rp{};
  rp.nson = ns;
  double l1 = 0, l2 = 0;
  for (int j = 0; j < ns; ++j) {
    const int s = e->children[e->child_off[root] + j];
    RootReparamSon& rs = rp.sons[j];
    rs.is_leaf = e->leaf_slot[s] >= 0;
    if (rs.is_leaf) {
      rs.codes = (const char*)e->d_codes + (size_t)e->leaf_slot[s] * N * e->code_bytes;
    } else {
      rs.lower = e->d_keep + (size_t)e->internal_idx[s] * clvn;
      rs.lower_exp = e->d_keep_exp + (size_t)e->internal_idx[s] * rows;
    }
    const size_t mo = ((size_t)pl * e->nn + s) * C * SS;
    rs.P = e->d_P + mo; rs.dP = e->d_dP + mo; rs.d2P = e->d_d2P + mo;
    if (j == 0) l1 = e->h_brlen[(size_t)point * e->nn + s];
    if (j == 1) l2 = e->h_brlen[(size_t)point * e->nn + s];
  }
  if (!(l1 + l2 > 0)) BPP_FAIL(BPPGPU_E_INVALID, "the two root branches have zero total length");
  rp.S = S; rp.C = C; rp.code_bytes = e->code_bytes; rp.N = N;
  rp.prow = e->clv_class_major ? 1 : C;
  rp.crow = e->clv_class_major ? N : 1;
  rp.len = l1 + l2;
  rp.pos = l1 / (l1 + l2);
  rp.code_table = e->d_code_table;
  rp.rootfreq = e->d_rootfreq_used + (size_t)point * S;
  rp.probs = e->d_probs; rp.weights = e->d_weights; rp.SR = e->d_SR; rp.rexp = e->d_rexp;
  const int grid = (int)((N + 127) / 128);
  double *d_part = nullptr, *d_out = nullptr;
  if (cudaMalloc(&d_part, (size_t)4 * grid * 8) != cudaSuccess || cudaMalloc(&d_out, 4 * 8) != cudaSuccess) {
    cudaFree(d_part); cudaFree(d_out);
    BPP_FAIL(BPPGPU_E_NOMEM, "out of device memory");
  }
  rp.part = d_part;
  cudaStream_t st = e->stream;
  root_reparam_kernel<<<grid, 128, 0, st>>>(rp);
  root_reparam_finalize_kernel<<<4, 256, 0, st>>>(d_part, grid, d_out);
  cudaError_t err = cudaGetLastError();
  if (err == cudaSuccess) err = cudaMemcpyAsync(out, d_out, 4 * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess) err = cudaStreamSynchronize(st);
  cudaFree(d_part); cudaFree(d_out);
  BPP_CUDA(err);
  return BPPGPU_OK;
}

int bppgpu_get_site_derivatives(bppgpu_engine* e, int32_t point, int32_t node, double* d1_out, double* d2_out) {
  ENGINE_SYNC(e);
  if (!d1_out || point < 0 || point >= e->npoints || node < 0 || node >= e->nn || node == e->root)
    BPP_FAIL(BPPGPU_E_INVALID, "bad point / node or null out");
  if (!e->keep) BPP_FAIL(BPPGPU_E_STATE, "bppgpu_get_site_derivatives needs BPPGPU_FLAG_KEEP_CLVS");
  if (e->path == PATH_POINTS) BPP_FAIL(BPPGPU_E_STATE, "not available on the batched-points path");
  if (point != e->last_point) BPP_FAIL(BPPGPU_E_STATE, "CLVs resident are those of point %d", e->last_point);
  if (!(e->last_want & BPPGPU_EVAL_D1) || !e->d_upper || !e->d_dP) BPP_FAIL(BPPGPU_E_STATE, "upper CLVs exist after an eval with derivatives");
  if (d2_out && (!(e->last_want & BPPGPU_EVAL_D2) || !e->d_d2P)) BPP_FAIL(BPPGPU_E_STATE, "second derivatives need an eval with BPPGPU_EVAL_D2");
  const int uslab = e->upper_slab[node];
  if (uslab < 0) BPP_FAIL(BPPGPU_E_STATE, "the upper CLV of tip %d is not materialised at this problem size", node);
  const int S = e->S, C = e->C;
  const long long N = e->N;
  if (N == 0) return BPPGPU_OK;
  const size_t clvn = (size_t)N * C * S, rows = (size_t)N * C, SS = (size_t)S * S;
  double *d_1 = nullptr, *d_2 = nullptr;
  if (cudaMalloc(&d_1, (size_t)N * 8) != cudaSuccess || (d2_out && cudaMalloc(&d_2, (size_t)N * 8) != cudaSuccess)) {
    cudaFree(d_1); cudaFree(d_2);
    cudaGetLastError();
    BPP_FAIL(BPPGPU_E_NOMEM, "out of device memory");
  }
  SiteDerivParams sp{};
  const bool leaf = e->leaf_slot[node] >= 0;
  sp.is_tip = leaf; sp.S = S; sp.C = C; sp.code_bytes = e->code_bytes;
  sp.nh_form = (e->flags & BPPGPU_FLAG_NH_DERIV) ? 1 : 0;
  sp.N = N;
  sp.prow = e->clv_class_major ? 1 : C;
  sp.crow = e->clv_class_major ? N : 1;
  const size_t mo = ((size_t)(point % e->pchunk) * e->nn + node) * C * SS;
  sp.P = e->d_P + mo; sp.dP = e->d_dP + mo; sp.d2P = d2_out ? e->d_d2P + mo : nullptr;
  sp.code_table = e->d_code_table;
  if (leaf) sp.codes = (const char*)e->d_codes + (size_t)e->leaf_slot[node] * N * e->code_bytes;
  else {
    sp.lower = e->d_keep + (size_t)e->internal_idx[node] * clvn;
    sp.lower_exp = e->d_keep_exp + (size_t)e->internal_idx[node] * rows;
  }
  sp.upper = e->d_upper + (size_t)uslab * clvn;
  sp.upper_exp = e->d_upper_exp + (size_t)uslab * rows;
  sp.SR = e->d_SR; sp.rexp = e->d_rexp; sp.probs = e->d_probs;
  sp.d1 = d_1; sp.d2 = d_2;
  cudaStream_t st = e->stream;
  site_deriv_kernel<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(sp);
  cudaError_t err = cudaGetLastError();
  if (err == cudaSuccess) err = cudaMemcpyAsync(d1_out, d_1, (size_t)N * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess && d2_out) err = cudaMemcpyAsync(d2_out, d_2, (size_t)N * 8, cudaMemcpyDeviceToHost, st);
  if (err == cudaSuccess) err = cudaStreamSynchronize(st);
  cudaFree(d_1); cudaFree(d_2);
  BPP_CUDA(err);
  return BPPGPU_OK;
}

int bppgpu_get_transition_probabilities(bppgpu_engine* e, int32_t point, int32_t node, unsigned which, double* out) {
  ENGINE_SYNC(e);
  if (point < 0 || point >= e->npoints || node < 0 || node >= e->nn || node == e->root || !out)
    BPP_FAIL(BPPGPU_E_INVALID, "bad point / node or null out");
  if (e->last_want == 0) BPP_FAIL(BPPGPU_E_STATE, "no evaluation yet");
  const int last_chunk0 = ((e->npoints - 1) / e->pchunk) * e->pchunk;
  if (point < last_chunk0) BPP_FAIL(BPPGPU_E_STATE, "tables resident are those of points >= %d", last_chunk0);
  const double* src = which == BPPGPU_WANT_P ? e->d_P : which == BPPGPU_WANT_DP ? e->d_dP : which == BPPGPU_WANT_D2P ? e->d_d2P : nullptr;
  if (!src) BPP_FAIL(BPPGPU_E_STATE, "requested table was not built by the last eval");
  if (which == BPPGPU_WANT_DP && !(e->last_want & BPPGPU_EVAL_D1)) BPP_FAIL(BPPGPU_E_STATE, "dP not built by the last eval");
  if (which == BPPGPU_WANT_D2P && !(e->last_want & BPPGPU_EVAL_D2)) BPP_FAIL(BPPGPU_E_STATE, "d2P not built by the last eval");
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  const size_t per = (size_t)e->C * e->S * e->S;
  BPP_CUDA(cudaMemcpy(out, src + ((size_t)(point - last_chunk0) * e->nn + node) * per, per * 8, cudaMemcpyDeviceToHost));
  return BPPGPU_OK;
}

int bppgpu_get_root_freqs(bppgpu_engine* e, int32_t point, double* out) {
  ENGINE_SYNC(e);
  if (point < 0 || point >= e->npoints || !out) BPP_FAIL(BPPGPU_E_INVALID, "bad point or null out");
  BPP_CUDA(cudaStreamSynchronize(e->stream));
  BPP_CUDA(cudaMemcpy(out, e->d_rootfreq_used + (size_t)point * e->S, e->S * 8, cudaMemcpyDeviceToHost));
  return BPPGPU_OK;
}

// ---- multi-GPU ------------------------------------------------------------------------------
int bppgpu_comm_unique_id(void* id_out) {
  if (!id_out) BPP_FAIL(BPPGPU_E_INVALID, "null id_out");
  NcclApi& api = nccl_api();
  if (!api.ok) BPP_FAIL(BPPGPU_E_NCCL, "libnccl.so.2 could not be loaded: %s", dlerror() ? dlerror() : "missing symbols");
  ncclUniqueId id;
  BPP_NCCL(api.GetUniqueId(&id));
  static_assert(sizeof(ncclUniqueId) == BPPGPU_UNIQUE_ID_BYTES, "unique id size");
  memcpy(id_out, &id, sizeof(id));
  return BPPGPU_OK;
}

int bppgpu_comm_init(bppgpu_engine* e, int32_t rank, int32_t nranks, const void* unique_id) {
  ENGINE_SYNC(e);
  if (!unique_id || nranks < 1 || rank < 0 || rank >= nranks) BPP_FAIL(BPPGPU_E_INVALID, "bad rank / nranks or null id");
  if (e->comm) BPP_FAIL(BPPGPU_E_STATE, "the engine already has a communicator");
  NcclApi& api = nccl_api();
  if (!api.ok) BPP_FAIL(BPPGPU_E_NCCL, "libnccl.so.2 could not be loaded: %s", dlerror() ? dlerror() : "missing symbols");
  ncclUniqueId id;
  memcpy(&id, unique_id, sizeof(id));
  ncclComm_t comm = nullptr;
  BPP_NCCL(api.CommInitRank(&comm, nranks, id, rank));
  e->comm = comm;
  e->comm_rank = rank;
  e->comm_nranks = nranks;
  if (nranks > 1) {
    cudaFree(e->d_wr_recs);
    e->d_wr_recs = nullptr;
    BPP_CUDA(dev_alloc(e, &e->d_wr_recs, (size_t)nranks * (e->S + 1)));
  }
  e->last_point = -1;
  return BPPGPU_OK;
}

int bppgpu_comm_finalize(bppgpu_engine* e) {
  ENGINE_SYNC(e);
  if (e->comm) BPP_NCCL(nccl_api().CommDestroy((ncclComm_t)e->comm));
  e->comm = nullptr;
  e->comm_rank = 0;
  e->comm_nranks = 1;
  return BPPGPU_OK;
}

int bppgpu_eval_status(bppgpu_engine* e, int32_t* numeric_failure) {
  ENGINE_SYNC(e);
  if (!numeric_failure) BPP_FAIL(BPPGPU_E_INVALID, "null argument");
  int status = 0;
  if (e->status_armed) BPP_CUDA(cudaMemcpy(&status, e->d_status, 4, cudaMemcpyDeviceToHost));
  *numeric_failure = status;
  if (status) BPP_FAIL(BPPGPU_E_NUMERIC, "ChromosomeSubstitutionModel: Taylor series did not reach convergence!");
  return BPPGPU_OK;
}

int bppgpu_eval_multi(bppgpu_engine* const* engines, int32_t n_engines, unsigned want, double* lnl, double* d1, double* d2) {
  if (!engines || n_engines < 1 || !engines[0]) BPP_FAIL(BPPGPU_E_INVALID, "no engines");
  const int nn = engines[0]->nn, np = engines[0]->npoints;
  for (int k = 0; k < n_engines; ++k) {
    if (!engines[k] || engines[k]->nn != nn || engines[k]->npoints != np)
      BPP_FAIL(BPPGPU_E_INVALID, "engine %d does not share the topology / number of points of engine 0", k);
    if (engines[k]->comm && engines[k]->comm_nranks > 1)
      BPP_FAIL(BPPGPU_E_STATE, "engine %d belongs to an NCCL job: its evaluations already return the job's totals", k);
    if (engines[k]->flags & BPPGPU_FLAG_WEIGHTED_ROOT)
      BPP_FAIL(BPPGPU_E_INVALID, "weighted root frequencies over pattern shards need the NCCL job form (bppgpu_comm_init)");
  }
  // enqueue every shard on its own device and stream, then collect: the shards run concurrently
  for (int k = 0; k < n_engines; ++k) {
    bppgpu_engine* e = engines[k];
    BPP_CUDA(cudaSetDevice(e->dev));
    int rc = eval_impl(e, want, e->stream, false);
    if (rc) return rc;
  }
  const size_t row = (size_t)(1 + 2 * nn);
  std::vector<double> tot((size_t)np * row, 0.0), h((size_t)np * row);
  for (int k = 0; k < n_engines; ++k) {
    bppgpu_engine* e = engines[k];
    BPP_CUDA(cudaSetDevice(e->dev));
    BPP_CUDA(cudaStreamSynchronize(e->stream));
    BPP_CUDA(cudaMemcpy(h.data(), e->d_out, h.size() * 8, cudaMemcpyDeviceToHost));
    int status = 0;
    if (e->status_armed) BPP_CUDA(cudaMemcpy(&status, e->d_status, 4, cudaMemcpyDeviceToHost));
    if (status) BPP_FAIL(BPPGPU_E_NUMERIC, "ChromosomeSubstitutionModel: Taylor series did not reach convergence!");
    for (size_t i = 0; i < tot.size(); ++i) tot[i] += h[i];   // shard order: deterministic
  }
  const unsigned lw = engines[0]->last_want;
  for (int p = 0; p < np; ++p) {
    const double* r = tot.data() + (size_t)p * row;
    if (lnl) lnl[p] = r[0];
    if (d1 && (lw & BPPGPU_EVAL_D1)) std::copy(r + 1, r + 1 + nn, d1 + (size_t)p * nn);
    if (d2 && (lw & BPPGPU_EVAL_D2)) std::copy(r + 1 + nn, r + 1 + 2 * nn, d2 + (size_t)p * nn);
  }
  return BPPGPU_OK;
}

int bppgpu_get_frontier_nodes(bppgpu_engine* e, int32_t* out) {
  if (!e || !out) BPP_FAIL(BPPGPU_E_INVALID, "null argument");
  *out = e->w4c_frontier_nodes;
  return BPPGPU_OK;
}

int bppgpu_get_stats(bppgpu_engine* e, bppgpu_stats* out) {
  if (!e || !out) BPP_FAIL(BPPGPU_E_INVALID, "null argument");
  e->stats.hbm_bytes_resident = (int64_t)e->bytes_resident;
  // collect the pruning-kernel timings recorded since the last call (waits for them to complete)
  e->stats.prune_ms_sum = 0.0;
  e->stats.prune_count = 0;
  cudaSetDevice(e->dev);
  for (int k = 0; k < e->ring_n; ++k) {
    const int i = (e->ring_head + bppgpu_engine::kRing - 1 - k) % bppgpu_engine::kRing;
    float ms = 0.f;
    if (cudaEventSynchronize(e->ring_b[i]) == cudaSuccess && cudaEventElapsedTime(&ms, e->ring_a[i], e->ring_b[i]) == cudaSuccess) {
      e->stats.prune_ms_sum += ms;
      e->stats.prune_count++;
    }
  }
  e->ring_n = 0;
  e->stats.pt_ms_sum = 0.0;
  e->stats.pt_count = 0;
  for (int k = 0; k < e->ptring_n; ++k) {
    const int i = (e->ptring_head + bppgpu_engine::kRing - 1 - k) % bppgpu_engine::kRing;
    float ms = 0.f;
    if (cudaEventSynchronize(e->ptring_b[i]) == cudaSuccess && cudaEventElapsedTime(&ms, e->ptring_a[i], e->ptring_b[i]) == cudaSuccess) {
      e->stats.pt_ms_sum += ms;
      e->stats.pt_count++;
    }
  }
  e->ptring_n = 0;
  cudaGetLastError();
  *out = e->stats;
  return BPPGPU_OK;
}

