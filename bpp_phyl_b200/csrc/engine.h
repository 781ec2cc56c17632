// Host-side engine state behind the opaque bppgpu_engine handle.
#pragma once
#include <cuda_runtime.h>

#include <string>
#include <vector>

#include "../../include/bppgpu.h"
#include "deriv_kernels.cuh"
#include "dmma_deriv_kernels.cuh"
#include "dmma_family_kernels.cuh"
#include "dmma_node_kernels.cuh"
#include "generic_kernels.cuh"
#include "points_kernels.cuh"
#include "chr_factored_kernels.cuh"
#include "pt_dmma_kernels.cuh"
#include "pt_kernels.cuh"
#include "walk_kernels.cuh"
#include "walk4c_kernels.cuh"

namespace bppgpu {

enum PathKind { PATH_NONE = 0, PATH_WALK4 = 1, PATH_WALKS = 2, PATH_GENERIC = 3, PATH_DMMA = 4, PATH_POINTS = 5 };

struct DevModel {
  // one device slab per model slot, allocated at the first upload and overwritten by later ones (an optimiser re-sends a model
  // of the same shape at every step): [V | Vinv | re | im | role | Q | Q2];  V .. role point into it
  double* slab = nullptr;
  double *V = nullptr, *Vinv = nullptr, *re = nullptr, *im = nullptr, *Q = nullptr, *Q2 = nullptr;
  double *Vp = nullptr, *Vinvp = nullptr, *rep = nullptr, *imp = nullptr;  // what the tensor-core P(t) kernel reads: V .. itself, or
  double* pslab = nullptr;                                                 // the padded / pair-permuted copies in `pslab` (S % 8, complex)
  bool has_Q = false;
  int* role = nullptr;
  double rate = 1.0, eps = 1e-4;
  unsigned flags = 0;
  int has_complex = 0;
  bool set = false;
  int S = 0;
  double q_l1 = 0.0;  // sum |Q_ij| (ChromosomeSubstitutionModel::getFirstNorm)
};

// Post-order "program" of the pruning recursion: one Op per internal node.
struct Program {
  std::vector<Op> ops;
  std::vector<Child> childs;
  int nslots = 0;
  Op* d_ops = nullptr;
  Child* d_childs = nullptr;
};

}  // namespace bppgpu

struct bppgpu_engine {
  int dev = 0;
  cudaStream_t stream = nullptr;
  int S = 0, C = 0, nn = 0, root = 0, npoints = 1, nmodels = 1, ncodes = 0, code_bytes = 1;
  long long N = 0;
  unsigned flags = 0;
  // topology (host)
  std::vector<int> child_off, children, parent;
  std::vector<int> leaf_slot;     // node id -> leaf slot or -1
  std::vector<int> leaf_nodes;    // leaf slot -> node id
  std::vector<int> internal_idx;  // node id -> keep index or -1
  std::vector<int> preorder;      // fathers before sons
  int nl = 0, ni = 0;
  // device inputs
  void* d_codes = nullptr;        // [nl][N] tip codes
  double* d_code_table = nullptr; // [ncodes][S]
  int* d_code_single = nullptr;   // [ncodes] state of an indicator row or -1
  double* d_weights = nullptr;    // [N]
  double *d_rates = nullptr, *d_probs = nullptr;
  double* d_rootfreq = nullptr;       // [npoints][S] as given
  double* d_rootfreq_used = nullptr;  // [npoints][S] as used (WEIGHTED_ROOT overwrites)
  double* d_brlen = nullptr;          // [npoints][nn]
  int* d_branch_model = nullptr;      // [npoints][nn]
  int* d_leaf_nodes = nullptr;
  std::vector<bppgpu::DevModel> models;
  bppgpu::ModelDev* d_models = nullptr;
  bool models_dirty = true;
  int brlen_dirty_lo = 0, brlen_dirty_hi = 0;   // points whose branch lengths changed on the host since the last upload [lo, hi)
  bool homogeneous_points = true;  // every branch of a point uses the same model slot
  std::vector<double> h_rates, h_probs;
  std::vector<double> h_brlen;  // [npoints][nn]
  std::vector<int> h_branch_model;
  // tables, sized for `pchunk` points
  int pchunk = 1;
  double *d_P = nullptr, *d_dP = nullptr, *d_d2P = nullptr;
  double* d_tiptab = nullptr;
  double *d_dtiptab = nullptr, *d_d2tiptab = nullptr;  // tip tables of dP, d2P (DMMA derivative path)
  double* d_dLc = nullptr;                              // [N][C][2]
  std::vector<int> upper_slab;                          // node id -> slab of d_upper, or -1
  // per-father fused upper + derivative pass (dmma_family_kernels.cuh)
  bool family = false;
  bool prune64 = false;          // S = 64, C = 1: fragment-order pruning kernel (dmma_prune_kernel<64, ...>)
  int prune_cfg = 0;             // warps x ring depth of dmma_prune_kernel (BPPGPU_PRUNE_CFG)
  bool clv_class_major = false;  // CLV slabs are [class][pattern][state] (S = 20 fragment-order kernels only)
  std::vector<int> fam_mask;   // node id -> 1 when its branch is served by its father's family launch
  int* d_fam_mask = nullptr;
  double* d_fam_part = nullptr;  // [nn][2][fam_grid]
  double *d_fam_packA = nullptr, *d_fam_packS = nullptr, *d_fam_packL = nullptr, *d_fam_packT = nullptr;  // B operands in fragment order (family_pack_kernel)
  int fam_grid = 0, fam_ppc = 0;
  int n_upper_slabs = 0;
  // walk4 artefacts (everything in walk order, see walk_kernels.cuh)
  std::vector<unsigned long long> w4_desc;
  std::vector<int> w4_tip_order;
  std::vector<bppgpu::PackBlock> w4_blocks;
  size_t w4_stream_len = 0;  // doubles per point
  int w4_tstride = 0;
  int w4_pt = 1;  // patterns per thread
  unsigned long long* d_w4_desc = nullptr;
  int* d_w4_tip_order = nullptr;
  bppgpu::PackBlock* d_w4_blocks = nullptr;
  double* d_w4_stream = nullptr;       // [pchunk][w4_stream_len]
  unsigned char* d_codesT = nullptr;   // [N][w4_tstride]
  bool codesT_dirty = true;
  // walk4c (class-uniform, chunk-streamed walk; value-only engines): see walk4c_kernels.cuh
  bool w4c = false;
  bppgpu::Program prog4c;                  // walk program whose leaf pushes use the register slot
  bppgpu::W4cProgram w4c_prog;             // descriptor words + chunk records (passed as a kernel parameter)
  size_t w4c_stream_bytes = 0;             // nchunks * CH
  // launch plan: the pattern list is walked in one or two segments -- full waves of the widest CTAs, then the remainder with
  // narrower ones (fewer patterns per thread, more CTAs per SM) so that the last wave is short
  struct W4cSeg { int pt; long long pat0, pat_end; int grid; size_t codes_off; int part0; };
  std::vector<W4cSeg> w4c_segs;
  std::vector<bppgpu::Pack4cBlock> w4c_blocks;
  std::vector<int2> w4c_tip_order;          // code rows in consumption order: {leaf slot, -1} or a cherry's {son 0, son 1}
  std::vector<char> w4c_cherry;            // [nn] node is a folded cherry: a wide tip of prog4c (BPPGPU_W4C_FRONTIER=0: none)
  int w4c_frontier_nodes = 0;              // folded cherries of the walk4c program in use
  int w4c_CH = 0, w4c_nchunks = 0, w4c_pt = 2, w4c_nw = 8, w4c_max_tips = 16;
  unsigned char* d_w4c_stream = nullptr;   // [pchunk][nchunks][CH]
  bppgpu::Pack4cBlock* d_w4c_blocks = nullptr;
  int2* d_w4c_tip_order = nullptr;
  unsigned* d_w4c_counter = nullptr;       // CTAs done in the current evaluation (reset by the last one)
  unsigned char* d_codesC = nullptr;       // [grid][ntips][PPC] tip codes as the CTAs stage them
  // CLV storage (one point at a time)
  double* d_keep = nullptr;  // [ni][N][C][S]
  int* d_keep_exp = nullptr; // [ni][N][C]
  double* d_gstack = nullptr;
  int* d_gstack_exp = nullptr;
  double* d_upper = nullptr;  // [nn][N][C][S] generic derivative pass
  int* d_upper_exp = nullptr;
  // outputs
  double* d_SR = nullptr;        // [N] of the last evaluated point
  int* d_rexp = nullptr;
  double* d_site_lnl = nullptr;  // [npoints][N]
  double* d_partials = nullptr;
  double* d_partials2 = nullptr;
  int n_partials = 0;
  double* d_out = nullptr;  // [npoints][1+2nn]
  double* d_scratch = nullptr;  // series / unclamped-P scratch
  size_t scratch_elems = 0;
  int* d_status = nullptr;
  // schedule
  bppgpu::Program prog;   // walk program (REG / SLOT children)
  bppgpu::Program gprog;  // generic program (all internal children read from keep)
  std::vector<std::vector<bppgpu::Child>> sibs;  // per node: siblings, generic kinds
  bppgpu::Child* d_sibs = nullptr;
  std::vector<int> sib_off;
  std::vector<bppgpu::Child> sibs_flat;
  int path = bppgpu::PATH_NONE;
  bool keep = false;
  // state flags
  bool have_weights = false, have_rates = false, have_codes_all = false;
  std::vector<char> have_tip, have_brlen, have_rootfreq;
  int last_point = -1;  // point whose CLVs / SR are currently resident
  unsigned last_want = 0;
  // stats
  bppgpu_stats stats{};
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // ring of event pairs bracketing the pruning kernel(s) of point 0 of each eval, on the launching stream
  static constexpr int kRing = 64;
  cudaEvent_t ring_a[kRing] = {}, ring_b[kRing] = {};
  int ring_n = 0;  // pairs recorded since the last collection (capped at kRing)
  int ring_head = 0;
  // same for the K1 P(t) launches (one pair per chunk of points)
  cudaEvent_t ptring_a[kRing] = {}, ptring_b[kRing] = {};
  int ptring_n = 0, ptring_head = 0;
  size_t bytes_resident = 0;
  // batched points without P tables (chr_factored_kernels.cuh): one character, one rate class, many parameter points
  bool status_armed = false;        // the status word was cleared for the evaluation in flight
  bool rootfreq_used_stale = true;  // d_rootfreq_used must be refreshed from d_rootfreq
  bool chr_factored = false;
  // level-batched pruning launches of the fragment-order tensor-core kernels (dmma_prune_level_kernel)
  bool level_batch = false;
  bppgpu::DmmaPruneParams* d_prune_nodes = nullptr;   // [internal nodes], grouped by (level, kind of sons)
  struct PruneGroup { int kind, first, count, ctas_per_node; };
  std::vector<PruneGroup> prune_groups;
  const void* prune_nodes_sig[3] = {nullptr, nullptr, nullptr};   // buffers the cached descriptors point into
  bppgpu::DmmaFamilyParams* d_family_nodes = nullptr; // [internal nodes], grouped by (depth, kind of sons)
  std::vector<PruneGroup> family_groups;
  const void* family_nodes_sig[4] = {nullptr, nullptr, nullptr, nullptr};
  unsigned family_nodes_want = 0;
  bool tables_allocated = true;          // d_P / d_keep of the table route (allocated on demand for factored engines)
  std::vector<unsigned short> h_codes;   // [nl] the single pattern's tip codes (host copy)
  std::vector<int> h_code_single;        // [ncodes]
  std::vector<double> h_code_table;      // [ncodes][S]
  std::vector<int> chr_level_tile0;      // first tile of every level (+ end)
  int chr_ntiles = 0;
  bool chr_tiles_dirty = true;
  int *d_chr_tile_edges = nullptr, *d_chr_tile_kind = nullptr, *d_chr_leaf_state = nullptr, *d_child_off = nullptr, *d_children = nullptr;
  double* d_chr_leaf_vec = nullptr;      // [nn][S]
  double* d_chr_term = nullptr;          // [fchunk][nn][S]
  int* d_chr_term_exp = nullptr;         // [fchunk][nn]
  int fchunk = 0;                        // points per pass of the factored route
  int* d_chr_bad = nullptr;              // [npoints] guard verdicts
  double* d_chr_guardP = nullptr;        // [gchunk][3][S][S]
  bool chr_slab = false;                 // slab-streamed level kernels (TMA ring; dmma.cuh chr_gemm_slab)
  bool chr_slab_dirty = true;            // the slab-ordered copies must be rebuilt from the model slabs
  double* d_chr_aslab = nullptr;         // [nmodels][V^-1 | V | (V^-1)^T] slab-ordered copies + transpose
  int gchunk = 0;
  double* d_chr_probe_t = nullptr;       // [npoints][3]
  int* d_chr_probe_bm = nullptr;         // [npoints][3]
  bppgpu::ModelDev* d_models_noclamp = nullptr;
  // compact copies of the per-point inputs / outputs of the points on the table route ("bad" points), [nbad_cap][...]
  int nbad_cap = 0;
  int* d_bad_idx = nullptr;
  double *d_bad_brlen = nullptr, *d_bad_rootfreq = nullptr, *d_bad_rootfreq_used = nullptr, *d_bad_site_lnl = nullptr, *d_bad_out = nullptr;
  int* d_bad_branch_model = nullptr;
  std::vector<int> chr_bad;              // host copy of the last guard
  long long chr_factored_points = 0, chr_table_points = 0;   // of the last evaluation
  // multi-GPU (pattern shards, one engine per GPU): NCCL communicator of the job, set by bppgpu_comm_init
  void* comm = nullptr;           // ncclComm_t
  int comm_rank = 0, comm_nranks = 1;
  double* d_wr_recs = nullptr;    // [nranks][S + 1] weighted-root records (exponent, S sums), all-gathered
  static constexpr int kStageThreads = 8;
  double* h_stage = nullptr;        // pinned staging of bppgpu_set_models (two model images per packing thread)
  cudaStream_t stage_stream[kStageThreads] = {};
  cudaEvent_t stage_ev[kStageThreads][2] = {};
  cudaEvent_t eval_done = nullptr;  // recorded at the end of every evaluation on the evaluation's stream
  cudaStream_t last_stream = nullptr;
};
