/*
 * bppgpu.h -- C ABI of the B200-native tree-likelihood hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b): a C++ shim that keeps
 * the reference's class surface (bpp::TransitionModel::getPij_t ...,
 * bpp::R/DRHomogeneousTreeLikelihood, bpp::DRNonHomogeneousTreeLikelihood)
 * binds exactly these entry points; see INTEGRATION.md.  All functions are
 * extern "C", take plain pointers and sizes, never throw, and return a status
 * code; bppgpu_last_error() gives the message for the calling thread.
 *
 * There is no CPU fallback: every entry point that computes fails with
 * BPPGPU_E_CUDA when no sm_100a device is usable.
 *
 * Reference interfaces replaced (paths relative to src/Bpp/Phyl/ of
 * anatshafir1/bpp-phyl):
 *   Model/SubstitutionModel.h:233,240,247        getPij_t / getdPij_dt / getd2Pij_dt2
 *   Model/AbstractSubstitutionModel.cpp:426-641  generic eigen / block / Taylor forms
 *   Model/ChromosomeSubstitutionModel.cpp:808-1001  Chromosome P(t) family (clamp, P.Q, Q^2.P)
 *   Likelihood/AbstractHomogeneousTreeLikelihood.cpp:341-414   pxy_/dpxy_/d2pxy_ tables
 *   Likelihood/RHomogeneousTreeLikelihood.cpp:162-216,802-863  pruning + root reduction
 *   Likelihood/DRHomogeneousTreeLikelihood.cpp:170-186,287-454,483-719  DR passes, d1/d2
 *   Likelihood/DRNonHomogeneousTreeLikelihood.cpp:370-541,904-962      NH form, weighted root
 */
#ifndef BPPGPU_H
#define BPPGPU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- status codes (SURVEY.md 8b "Error conventions") ---------------------- */
enum {
  BPPGPU_OK = 0,
  BPPGPU_E_INVALID = 1, /* bad argument / shape                                */
  BPPGPU_E_STATE = 2,   /* call order: data, model, lengths not set yet ...    */
  BPPGPU_E_CUDA = 3,    /* CUDA runtime error, or no usable device             */
  BPPGPU_E_NCCL = 4,
  BPPGPU_E_NUMERIC = 5, /* e.g. Taylor series did not converge                 */
  BPPGPU_E_NOMEM = 6
};

/* message of the last failing call on this thread ("" if none) */
const char* bppgpu_last_error(void);
/* ABI version, bumped on incompatible change */
int bppgpu_abi_version(void);
/* number of visible CUDA devices (0 -> nothing below can compute) */
int bppgpu_device_count(int* n);
/* sizeof of the ABI structs as this library was compiled: which = 0 bppgpu_model_desc,
 * 1 bppgpu_config, 2 bppgpu_stats (lets a foreign-language binding verify its mirror) */
int bppgpu_sizeof(int which);

/* ---- site-pattern compression (host side, integer work, bit-exact) -------------
 * bpp::SitePatterns::SitePatterns (SitePatterns.cpp:52-106): sort the alignment columns by their
 * character string (Site::toString(), here the `col_bytes` bytes of each column in the sequence order
 * of the container), merge identical neighbours.  Outputs (caller-allocated, capacity n_sites):
 *   pattern_site[k]  original position of the site that represents pattern k (sites_)
 *   weights[k]       number of sites with pattern k (weights_)
 *   indices[i]       pattern of site i (indices_)
 * Patterns come out in lexicographic (memcmp) order of their column strings.                  */
int bppgpu_site_patterns(const uint8_t* columns, int64_t n_sites, int32_t col_bytes, int64_t* pattern_site,
                         uint32_t* weights, int64_t* indices, int64_t* n_patterns);

/* The same compression on the device (SURVEY 8f-4): columns are copied to the GPU, sorted there (one stable radix pass per
 * 8-byte word of the column, last word first), runs of identical columns numbered, and -- optionally -- the tip codes the
 * engine consumes extracted: tip_codes[l * n_patterns + k] = element l of the column of pattern k (elements of `code_bytes`
 * = 1 or 2 bytes, col_bytes / code_bytes leaves; caller-allocated, capacity n_sites * col_bytes bytes; NULL to skip), i.e.
 * row l is what bppgpu_set_tip_codes takes for leaf l.  Results are identical, bit for bit, to bppgpu_site_patterns.
 * `columns` and every output buffer may be pageable host memory (moved through pinned staging buffers by several host threads),
 * pinned / registered host memory (one direct DMA each) or DEVICE memory of `device` (device-to-device copies: nothing crosses PCIe).
 * No CPU fallback: BPPGPU_E_CUDA without a usable sm_100a device.                                                   */
int bppgpu_site_patterns_device(int device, const uint8_t* columns, int64_t n_sites, int32_t col_bytes, int32_t code_bytes,
                                int64_t* pattern_site, uint32_t* weights, int64_t* indices, int64_t* n_patterns,
                                void* tip_codes);

/* The R classes' recursive per-subtree compression (SURVEY 8 a4; host side, bit-exact integer work):
 * DRASRTreeLikelihoodData::initLikelihoodsWithPatterns (Likelihood/DRASRTreeLikelihoodData.cpp:218-332).  At every node the
 * father's unique columns are cut down to the node's own leaves (tree order) and compressed again; what comes out is
 *   n_patterns[n]                       number of distinct columns of the subtree below n (its likelihood-array length)
 *   links[link_offsets[s] + i]          pattern of son s that father pattern i reads = patternLinks_[father][s][i]
 *                                       (DRASRTreeLikelihoodData.h:145, getArrayPositions :231); n_patterns[father] entries,
 *                                       none for the root
 *   root_links[site], root_weights[k]   SitePatterns::getIndices / getWeights of the root's own compression.
 * columns: n_sites columns of n_seqs elements of elem_bytes bytes, in CONTAINER order; leaf_seq[node] = position of the
 * leaf's sequence inside a column (-1 for internal nodes).  n_patterns [n_nodes] and link_offsets [n_nodes + 1] are always
 * written; links / root_links / root_weights may be NULL (call once for the sizes, again with link_offsets[n_nodes] slots). */
int bppgpu_subtree_patterns(const uint8_t* columns, int64_t n_sites, int32_t n_seqs, int32_t elem_bytes, int32_t n_nodes,
                            const int32_t* child_offsets, const int32_t* children, int32_t root, const int32_t* leaf_seq,
                            int64_t* n_patterns, int64_t* link_offsets, int64_t* links, int64_t* root_links,
                            uint32_t* root_weights);

/* ---- model descriptor ------------------------------------------------------
 * What bpp::SubstitutionModel exposes (Model/SubstitutionModel.h:468-525):
 * getGenerator, getEigenValues, getIEigenValues, isDiagonalizable,
 * isNonSingular, getRowLeftEigenVectors, getColumnRightEigenVectors, getRate.
 * All matrices row-major S x S; x = from-state row, y = to-state column.     */
enum {
  BPPGPU_MODEL_DIAGONALIZABLE = 1u << 0, /* isDiagonalizable()                   */
  BPPGPU_MODEL_NONSINGULAR = 1u << 1,    /* isNonSingular()                      */
  BPPGPU_MODEL_CLAMP01 = 1u << 2,        /* Chromosome: P<0 -> 1e-20, P>1 -> 1   */
  BPPGPU_MODEL_CHR_DERIV = 1u << 3,      /* Chromosome: dP = P.Q.rate, d2P = Q^2.P.rate^2 */
  BPPGPU_MODEL_CHR_TAYLOR = 1u << 4,     /* Chromosome singular path: L1-norm scaling +
                                            the reference's 1e-4 truncation rule          */
  BPPGPU_MODEL_EXACT_EXPM = 1u << 5      /* singular path: run the series to FP64
                                            convergence instead of the reference's cut   */
};

typedef struct bppgpu_model_desc {
  int32_t n_states;
  uint32_t flags;
  double rate;               /* getRate()                                           */
  const double* right_eigen; /* V   [S*S] columns = right eigenvectors              */
  const double* left_eigen;  /* V^-1 [S*S] rows   = left eigenvectors               */
  const double* eigen_re;    /* [S]                                                  */
  const double* eigen_im;    /* [S] or NULL (all real)                               */
  const double* generator;   /* Q [S*S]; required unless DIAGONALIZABLE|NONSINGULAR  */
  double taylor_epsilon;     /* Chromosome truncation threshold (get_epsilon(), 1e-4)*/
} bppgpu_model_desc;

enum { BPPGPU_WANT_P = 1, BPPGPU_WANT_DP = 2, BPPGPU_WANT_D2P = 4 };

/* Interface 1: batched P(t) family for one model, host in / host out.
 * out arrays are [n_t][S][S]; pass NULL for tables not in `want`.
 * getPij_t(t) for a single t is n_t = 1.                                      */
int bppgpu_pt_batch(int device, const bppgpu_model_desc* model, int64_t n_t, const double* t,
                    unsigned want, double* P, double* dP, double* d2P);

/* ---- Interface 2: tree likelihood engine ----------------------------------- */
typedef struct bppgpu_engine bppgpu_engine;

enum {
  BPPGPU_FLAG_KEEP_CLVS = 1u << 0,   /* keep every node's lower CLV in HBM (needed for
                                        derivatives and bppgpu_get_clv)                 */
  BPPGPU_FLAG_R_SEMANTICS = 1u << 1, /* root reduction drops non-positive terms like the
                                        R classes (RHomogeneousTreeLikelihood.cpp:198,213);
                                        default = DR semantics (clamp SR<0 to 0)        */
  BPPGPU_FLAG_WEIGHTED_ROOT = 1u << 2, /* root frequencies = normalised per-state root
                                        likelihood (DRNonHomogeneousTreeLikelihood.cpp:927-962) */
  BPPGPU_FLAG_NH_DERIV = 1u << 3,    /* derivative in the NH numerator/denominator form
                                        (DRNonHomogeneousTreeLikelihood.cpp:370-413)    */
  BPPGPU_FLAG_FORCE_GENERIC = 1u << 4 /* run the unspecialised one-launch-per-node kernels
                                        (cross-check of the specialised paths)          */
};

typedef struct bppgpu_config {
  int32_t n_states;             /* S                                                   */
  int32_t n_cats;               /* C rate classes                                      */
  int64_t n_patterns;           /* N patterns held by THIS engine (a shard)            */
  int32_t n_nodes;              /* nodes of the flattened tree                         */
  int32_t root;                 /* id of the root node                                 */
  const int32_t* child_offsets; /* [n_nodes+1] CSR; a node with no children is a leaf  */
  const int32_t* children;      /* [child_offsets[n_nodes]] son ids in son order       */
  int32_t n_points;             /* independent parameter points evaluated per call     */
  int32_t n_models;             /* model slots (>=1)                                   */
  int32_t n_codes;              /* rows of code_table                                  */
  int32_t code_bytes;           /* 1 (uint8) or 2 (uint16) per tip code                */
  const double* code_table;     /* [n_codes][S]: getInitValue(s, code) (0/1 or probs)  */
  int32_t device;               /* CUDA device ordinal                                 */
  uint32_t flags;
} bppgpu_config;

int bppgpu_create(const bppgpu_config* cfg, bppgpu_engine** out);
int bppgpu_destroy(bppgpu_engine* e);

/* tip data: codes[N] for leaf `node` (copied) */
int bppgpu_set_tip_codes(bppgpu_engine* e, int32_t node, const void* codes);
/* all tips at once: codes[n_leaves][N], leaf rows in increasing node-id order
 * (bppgpu_leaf_slot gives the row of a leaf node)                             */
int bppgpu_set_all_tip_codes(bppgpu_engine* e, const void* codes);
int bppgpu_leaf_slot(bppgpu_engine* e, int32_t node, int32_t* slot);
/* pattern weights (SitePatterns::getWeights, unsigned int) */
int bppgpu_set_pattern_weights(bppgpu_engine* e, const uint32_t* w);
/* rate classes: getCategory(c), getProbability(c) */
int bppgpu_set_rates(bppgpu_engine* e, const double* rates, const double* probs);
/* model slot (eigensystem copied to the device) */
int bppgpu_set_model(bppgpu_engine* e, int32_t slot, const bppgpu_model_desc* m);
/* many slots at once (what an optimiser over a batch of parameter points sends every step): each model is packed into a
 * pinned staging image and copied asynchronously as ONE contiguous transfer, instead of several pageable copies          */
int bppgpu_set_models(bppgpu_engine* e, int32_t first_slot, int32_t n, const bppgpu_model_desc* descs);
/* per point: model slot of the branch above each node (default: slot 0, or slot
 * `point` when n_models == n_points)                                           */
int bppgpu_set_branch_models(bppgpu_engine* e, int32_t point, const int32_t* slot_of_node);
/* per point: length of the branch above each node, indexed by node id; the
 * root's entry is ignored.  `t` is copied before the call returns; the device copy
 * is refreshed by the next evaluation, one transfer for all points set since the
 * previous one (an optimiser over thousands of points sets them one by one)      */
int bppgpu_set_branch_lengths(bppgpu_engine* e, int32_t point, const double* t);
/* per point: root frequencies [S] */
int bppgpu_set_root_freqs(bppgpu_engine* e, int32_t point, const double* pi);

enum { BPPGPU_EVAL_LNL = 1, BPPGPU_EVAL_D1 = 2, BPPGPU_EVAL_D2 = 4 };

/* One full evaluation for every point: P(t) tables for all branches, pruning,
 * root reduction [, prefix pass and branch derivatives].
 * lnl[n_points]; d1, d2 [n_points][n_nodes] = d(lnL)/dt and the reference's
 * sum_i w_i (d2L_i/L_i - (dL_i/L_i)^2), i.e. derivatives of +lnL; the shim
 * flips the sign for getFirstOrderDerivative (DRHomogeneousTreeLikelihood.cpp:367). */
int bppgpu_eval(bppgpu_engine* e, unsigned want, double* lnl, double* d1, double* d2);

/* Same, results left in device memory as [n_points][1 + 2*n_nodes] doubles
 * (lnL, d1[n_nodes], d2[n_nodes]) at `dev_out`, enqueued on `cuda_stream`
 * (a cudaStream_t; NULL = the engine's stream) without a host sync, so the
 * caller can follow with an NCCL all-reduce on the same stream.               */
int bppgpu_eval_device(bppgpu_engine* e, unsigned want, double* dev_out, void* cuda_stream);

/* accessors (valid after an eval) */
int bppgpu_get_site_lnl(bppgpu_engine* e, int32_t point, double* out /* [N] */);
/* which: 0 = lower (subtree) CLV of `node`, 1 = upper (rest of tree, conditional on
 * the father's state).  clv [N][C][S] in the reference's VVVdouble order, values
 * are scaled per (pattern, class) row: true = clv[i][c][.] * 2^-scale_exp[i][c]
 * (scale_exp is [N][C]).  Needs BPPGPU_FLAG_KEEP_CLVS.                          */
int bppgpu_get_clv(bppgpu_engine* e, int32_t point, int32_t node, int32_t which, double* clv,
                   int32_t* scale_exp);
/* Consumers of the device-resident DR arrays (ancestral reconstruction, posterior rates), valid after an eval with
 * derivatives (the prefix pass must have run; the root needs only the value pass):
 *   likelihood_at_node [N][C][S] + scale_exp [N][C] = DRTreeLikelihood::computeLikelihoodAtNode(nodeId, VVVdouble&)
 *       (Likelihood/DRTreeLikelihood.h:92-102; DRHomogeneousTreeLikelihood::computeLikelihoodAtNode_,
 *        DRHomogeneousTreeLikelihood.cpp:723-815): true = value * 2^-scale_exp[i][c];
 *   posterior [N][C][S] = DRTreeLikelihoodTools::getPosteriorProbabilitiesForEachStateForEachRate(drl, nodeId)
 *       (Likelihood/DRTreeLikelihoodTools.cpp:46-119), as read by MarginalAncestralStateReconstruction.
 * Any of the three outputs may be NULL.  For a leaf whose upper CLV is not materialised (large problems) only
 * `posterior` is available (the reference's leaf formula needs the leaf likelihoods alone).                      */
int bppgpu_get_node_posteriors(bppgpu_engine* e, int32_t point, int32_t node, double* likelihood_at_node,
                               int32_t* scale_exp, double* posterior);
/* MarginalNonRevAncestralStateReconstruction (fork; Likelihood/MarginalNonRevAncestralStateReconstruction.h:66-207, .cpp:10-136)
 * for one node, from the device-resident lower / upper arrays:
 *   posterior [N][S]    = postProbNode_[node][i][x]: P(state at node = x | data of distinct site i)
 *       (computePosteriorProbabilitiesOfNodesForEachStatePerSite, .cpp:10-48; root: getRootPosteriorProb, :139-153)
 *   joint [N][S][S]     = jointProbabilities_[node][i][x][y]: P(node = x, father = y | data)
 *       (getJointLikelihoodFatherNode, .cpp:52-88, summed over the root states); NULL to skip; must be NULL at the root.
 * The reference's loop over the S root states with DRNonHomogeneousTreeLikelihood::computeLikelihoodPrefixConditionalOnRoot
 * (DRNonHomogeneousTreeLikelihood.cpp:1026-1162) collapses to the ordinary prefix arrays (linearity in the root state), so this
 * is one pass.  Valid after an eval with BPPGPU_EVAL_D1 on an engine created with BPPGPU_FLAG_KEEP_CLVS (the root needs
 * the value pass only).                                                                                              */
int bppgpu_get_marginal_posteriors(bppgpu_engine* e, int32_t point, int32_t node, double* posterior, double* joint);
/* MLAncestralStateReconstruction (fork; Likelihood/MLAncestralStateReconstruction.h, .cpp:6-188, leaf arrays
 * DRASRTreeLikelihoodData.cpp:265-300): joint maximum-likelihood reconstruction (Pupko et al. 2000) with the transition
 * probabilities and root frequencies of the last evaluation -- a max-product pass up the tree, the best root state of class 0,
 * and the trace back (getAllAncestralStates, .cpp:136-186), all on the device.
 *   states [n_nodes][N] int32   state of every node (a leaf: its observed state) per distinct site
 *   best_lnl [N] or NULL        log of the joint likelihood of that assignment (class 0): log max_x pi_x prod ...
 * Like the reference the traceback tables are those of the LAST rate class and the root uses class 0 (it "assumes one class");
 * unlike it, rows are rescaled by powers of two, so large trees do not underflow.                                          */
int bppgpu_ml_ancestral_states(bppgpu_engine* e, int32_t point, int32_t* states, double* best_lnl);
/* Derivatives of lnL with respect to "BrLenRoot" = l1 + l2 and "RootPosition" = l1 / (l1 + l2), the re-parametrisation of
 * the two root branches of a rooted tree (reparametrizeRoot; AbstractNonHomogeneousTreeLikelihood.cpp:319-330, :386-389):
 *   out[0..3] = d lnL / d BrLenRoot, d lnL / d RootPosition, d2 lnL / d BrLenRoot^2, d2 lnL / d RootPosition^2
 * = minus DRNonHomogeneousTreeLikelihood::getFirstOrderDerivative / getSecondOrderDerivative of those two names
 * (DRNonHomogeneousTreeLikelihood.cpp:445-478, :576-867).  The root's first two sons are root1, root2; valid after an
 * eval with BPPGPU_EVAL_D2 (dP, d2P and the lower arrays resident).                                                   */
int bppgpu_get_root_reparam_derivatives(bppgpu_engine* e, int32_t point, double out[4]);
/* DRASDRTreeLikelihoodData::getDLikelihoodArray(nodeId) / getD2LikelihoodArray(nodeId) (filled by
 * DRHomogeneousTreeLikelihood::computeTreeDLikelihoodAtNode / computeTreeD2LikelihoodAtNode, DRHomogeneousTreeLikelihood.cpp:
 * 287-326, :373-411): per pattern, (dL_i / d t_node) / L_i and (d2L_i / d t_node^2) / L_i, computed on the device from the
 * resident lower / upper arrays after an eval with derivatives.  d2_out may be NULL.                                      */
int bppgpu_get_site_derivatives(bppgpu_engine* e, int32_t point, int32_t node, double* d1_out /* [N] */, double* d2_out /* [N] */);
/* which: BPPGPU_WANT_P / _DP / _D2P; out [C][S][S] = pxy_[node][c][x][y] */
int bppgpu_get_transition_probabilities(bppgpu_engine* e, int32_t point, int32_t node,
                                        unsigned which, double* out);
/* root frequencies actually used (differs from the input with WEIGHTED_ROOT) */
int bppgpu_get_root_freqs(bppgpu_engine* e, int32_t point, double* out /* [S] */);

/* introspection for benches/tests */
typedef struct bppgpu_stats {
  int64_t kernel_launches; /* kernels launched by the last eval                   */
  int64_t clv_updates;     /* (node,pattern,cat,state) elements produced by it    */
  double last_eval_ms;     /* device time of the last bppgpu_eval (CUDA events)   */
  double prune_ms;         /* ... of its pruning kernel(s) (point 0)              */
  double prune_ms_sum;     /* pruning-kernel device time summed over the evals    */
  int64_t prune_count;     /* ... since the previous bppgpu_get_stats (max 64)    */
  double pt_ms_sum;        /* device time of the K1 P(t) launches, same window    */
  int64_t pt_count;        /* number of K1 launch groups timed (one per chunk)    */
  int64_t hbm_bytes_resident;
  int32_t stack_slots;
  int32_t path;            /* which kernel family ran (see DESIGN.md)             */
  int64_t factored_points; /* batched-points engines, last eval: points evaluated
                              without P tables (chr_level_kernel) ...             */
  int64_t table_points;    /* ... and points the guard sent to the table route    */
  int32_t chr_tiles_tip;   /* column tiles per point: observed-tip tiles (one GEMM) */
  int32_t chr_tiles_dense; /* ... and dense tiles (two GEMMs)                     */
  int32_t chr_cblocks_tip;  /* 8-column blocks in use over the tip tiles (a tile runs only those through the tensor cores) */
  int32_t chr_cblocks_dense; /* ... and over the dense tiles                       */
} bppgpu_stats;
int bppgpu_get_stats(bppgpu_engine* e, bppgpu_stats* out);
/* DNA walk (value-only S = 4 engines): cherries folded into wide tip tables, i.e. evaluated once per tip-code pair instead of
 * once per pattern (0 when none is; BPPGPU_W4C_FRONTIER=0 at engine creation folds none) */
int bppgpu_get_frontier_nodes(bppgpu_engine* e, int32_t* out);

/* ---- multi-GPU: site patterns shard, nothing else does (SURVEY 8e) ---------------------------------------------------
 * The pattern loop of RHomogeneousTreeLikelihood::computeSubtreeLikelihood (RHomogeneousTreeLikelihood.cpp:839-861) has no
 * dependence between patterns, so every GPU holds one engine over a contiguous block of the compressed pattern list (its own
 * tip codes and weights; tree, models, rates and branch lengths replicated) and the only exchange is the sum of the per-shard
 * (lnL, d1[], d2[]) rows -- plus, with BPPGPU_FLAG_WEIGHTED_ROOT, one (exponent, S sums) record per shard before the root
 * reduction (DRNonHomogeneousTreeLikelihood.cpp:927-962 sums over ALL sites).
 *
 * (a) one process per GPU (MPI / torchrun): NCCL inside the engine.  Rank 0 calls bppgpu_comm_unique_id and distributes
 *     the 128 bytes by its own means; every rank calls bppgpu_comm_init on its engine.  From then on bppgpu_eval and
 *     bppgpu_eval_device all-reduce their result rows on the evaluation's stream (all ranks must call them in the same
 *     order) and return the whole alignment's lnL / d1 / d2 on every rank.  libnccl.so.2 is loaded at the first call; a
 *     process that already has an NCCL (torch) shares it.  Errors: BPPGPU_E_NCCL.
 * (b) one process driving several GPUs: create one engine per device and call bppgpu_eval_multi, which enqueues every
 *     shard on its own device and stream, waits, and adds the rows on the host in shard order.                          */
#define BPPGPU_UNIQUE_ID_BYTES 128
int bppgpu_comm_unique_id(void* id_out /* [BPPGPU_UNIQUE_ID_BYTES] */);
int bppgpu_comm_init(bppgpu_engine* e, int32_t rank, int32_t nranks, const void* unique_id);
int bppgpu_comm_finalize(bppgpu_engine* e);
int bppgpu_eval_multi(bppgpu_engine* const* engines, int32_t n_engines, unsigned want, double* lnl, double* d1, double* d2);
/* After bppgpu_eval_device (which never synchronises): waits for that evaluation and reports its numeric status -- 0, or
 * BPPGPU_E_NUMERIC with *numeric_failure = 1 where the reference throws "Taylor series did not reach convergence".        */
int bppgpu_eval_status(bppgpu_engine* e, int32_t* numeric_failure);

/* ---- host-side utilities (not on the evaluation path) ----------------------------------------------------------------
 * bppgpu_host_model: build a named model with the C++ host code of this library -- the generator of the model class and
 * AbstractSubstitutionModel::updateMatrices (Model/AbstractSubstitutionModel.cpp:175-421; Chromosome:
 * Model/ChromosomeSubstitutionModel.cpp:431-802) -- and copy out what bppgpu_model_desc needs.  Names and parameter lists:
 *   "GTR" a b c d e piA piC piG piT (Model/Nucleotide/GTR.cpp:84-124)   "HKY85" kappa piA piC piG piT   "T92" kappa theta
 *   "K80" kappa   "JC69"   "LG08" (Model/Protein/LG08.cpp)   "YN98" kappa omega (Model/Codon/YN98.cpp:51-77)
 *   "GY94" kappa V (Model/Codon/GY94.cpp:49-71, Grantham distances)
 *   "Chromosome" min max gain loss dupl demi [gainR lossR duplR baseNum baseNumR maxChrRange]
 * Missing trailing parameters take the class defaults.  Output arrays are caller-allocated ([S*S] / [S]); any may be NULL.
 * Call once with all arrays NULL to learn *n_states.                                                                  */
int bppgpu_host_model(const char* name, const double* params, int32_t n_params, int32_t* n_states, uint32_t* flags, double* rate,
                      double* Q, double* V, double* Vinv, double* eigen_re, double* eigen_im, double* freq);
/* FP64 ceilings of `device` measured now: DFMA (CUDA-core FP64 pipe) and DMMA mma.sync m8n8k4 (the FP64 tensor path of
 * sm_100a), in TFLOP/s.  About 0.2 s.                                                                                   */
int bppgpu_measure_fp64_peak(int device, double* dfma_tflops, double* dmma_tflops);

#ifdef __cplusplus
}
#endif
#endif /* BPPGPU_H */
