// K2 + K3 for S = 4 (DNA), value-only evaluations: the CLASS-UNIFORM, CHUNK-STREAMED tree walk.
//
// Same idea as walk4_kernel (walk_kernels.cuh): the pruning recursion (RHomogeneousTreeLikelihood::computeSubtreeLikelihood,
// Likelihood/RHomogeneousTreeLikelihood.cpp:802-863; DR twin DRHomogeneousTreeLikelihood.cpp:483-539, :819-864) is independent
// per (pattern, rate class) row, so one launch walks the whole post-order program and every CLV stays on chip; the root
// reduction (RHomogeneousTreeLikelihood.cpp:162-216 / DRHomogeneousTreeLikelihood.cpp:653-719) is fused.
//
// What ncu showed on walk4_kernel (profiles/r1_final_walk4_pt2_ncu_summary.csv): l1tex data-pipe wavefronts 82.6 %, FP64 pipe
// 24 %, long-scoreboard stalls 4.4 per issue -- every thread fetched the 128-byte P block of its class from global memory for
// each internal child (32 wavefronts per warp for 2 patterns), tip rows and the shared-memory stack went through the same pipe.
// This kernel removes that traffic instead of hiding it:
//   * a warp is CLASS-UNIFORM (32 lanes = 32 x PT patterns of ONE rate class), so P of a child is the same 16 doubles for
//     the whole warp: 8 broadcast LDS.128 (1 wavefront each) instead of 4 LDG.256 x 8 wavefronts;
//   * the walk's tables (P blocks, per-branch tip tables, op descriptors) are cut into fixed-size CHUNKS in walk order and
//     streamed L2 -> shared memory by the TMA engine (cp.async.bulk + mbarrier full/empty ring, one elected producer thread):
//     no dependent global load is left on the critical path, the chunk after next is always in flight;
//   * a tip row is a gather from a 128-byte [code][4] table in shared memory: every bank holds one address, 2 LDS.128;
//   * the innermost level of the CLV stack lives in REGISTERS: a push whose lifetime contains no other push ("leaf push":
//     the sibling evaluated next is a caterpillar) writes its result to the second register set `w`, and the father reads it
//     from there; only deeper pushes go to the shared-memory stack (two 16-byte planes: conflict free);
//   * tip codes are read coalesced: codes8[group of 8 tips][pattern] (one 8-byte word per pattern and 8 tips).
// Arithmetic, multiplication order and rescaling rule are those of walk4_kernel: the two kernels agree bit for bit per site.
#pragma once
#include "walk_kernels.cuh"

namespace bppgpu {

constexpr int kW4cMaxWarps = 8;           // warps per CTA: 8 (two CTAs per SM at 128 registers) or 4 (three at 168)
constexpr int kW4cStages = 3;
constexpr int kW4cMaxTipsPerChunk = 16;   // tip-code rows staged with a chunk
constexpr int kW4cMaxOps = 3072;          // descriptors (8 bytes each) that fit the kernel-parameter block
constexpr int kW4cMaxChunks = 1024;
constexpr int kW4cMaxWideCodes = 64;      // code pairs of a folded cherry (ncodes <= 8)

// W4C_CHERRY only names a table block (Pack4cBlock::kind): the walk reads a cherry as a wide tip
enum W4cKind { W4C_TIP = 0, W4C_SLOT = 1, W4C_REG = 2, W4C_RSL = 3, W4C_CHERRY = 4 };
// binary shapes (the only ones a bifurcating tree's planner emits); 0 = generic child loop
// one-hot shape bits (tested one by one: the dispatch stays a chain of uniform branches).  W4C_WA / W4C_WB: the first / second
// tip block the handler consumes is a wide tip (a folded cherry, below)
enum W4cShape { W4C_GENERIC = 0, W4C_TS = 1 /* tip + current rows */, W4C_TT = 2, W4C_JW = 4 /* register slot + current rows */,
                W4C_JS = 8 /* shared-memory slot + current rows */, W4C_DSTW = 16 /* result goes to the register slot */,
                W4C_WA = 32, W4C_WB = 64 };

// Folded cherries.  The conditional likelihood of a cherry (an internal node whose two sons are tips) depends on the pair of
// tip codes only, so the table pass evaluates it once per code pair -- tip terms, product, rescale, and the father's term
// P_cherry . l -- and the walk reads the result like a tip: a WIDE TIP with W = ncodes^2 codes (code_a * ncodes + code_b)
// and an exponent per row.  Block layout: [class][W][4] doubles, then [class][W] int32 exponents.  Every step is the walk's own
// arithmetic (the functions below are shared by both kernels), so a folded cherry gives the walk's bits.
__host__ __device__ inline int w4c_wide_block_bytes(int C, int W) { return (C * W * 36 + 15) & ~15; }

// P . l for one row x of P: the association of every tip table and of term_internal
__device__ __forceinline__ double w4c_dot(double p0, double p1, double p2, double p3, double l0, double l1, double l2, double l3) {
  return fma(p3, l3, fma(p2, l2, fma(p1, l1, p0 * l0)));
}
__device__ __forceinline__ int w4c_max_hi(const double (&a)[4]) {
  return max(max(hi_word(a[0]), hi_word(a[1])), max(hi_word(a[2]), hi_word(a[3])));
}
// the power-of-two rescale of one row whose largest high word is m
__device__ __forceinline__ void w4c_rescale(double (&a)[4], int m, int& e) {
  if (m < kScaleThresholdHi && m >= (1 << 20)) {
    const int k = rescale_shift(m);
    const double f = pow2(k);
    a[0] *= f; a[1] *= f; a[2] *= f; a[3] *= f;
    e += k;
  }
}

// The walk program lives in the KERNEL PARAMETER block (constant bank, up to 32 KB since CUDA 12.1): descriptors and chunk
// records are read with warp-uniform loads and the per-op dispatch runs on the uniform datapath -- no convergence barriers, no
// shared-memory round trip for the descriptor.
//   descriptor .x: bits 0-3 one-hot shape (none = generic), bit 4 result goes to the register slot, bits 8-13 shared slot that
//   also receives the result when bit 14 is set, bits 16-21 the shared slot read by W4C_JS, bits 24-27 nchild;
//   .y (generic ops): bits 0-11 child kinds (2 bits each, son order), bits 12-31 the slots of its W4C_SLOT children (6 bits each)
//   chunk record: bits 0-15 first tip (consumption order) of the chunk, bits 16-20 number of tips, bits 21-25 number of ops
struct W4cProgram {
  uint2 desc[kW4cMaxOps];
  unsigned chunk[kW4cMaxChunks];
};

struct Walk4cParams {
  const unsigned char* stream;       // [nchunks][CH] this point's table chunks
  const unsigned char* codesC;       // [gridDim.x][ntips][PPC] tip codes, consumption order, one byte per pattern
  int nchunks, CH, nslots, ncodes, ntips;
  int wide_codes;                    // codes of a wide tip (folded cherry): ncodes^2
  int max_tips;                      // tip-code rows a ring stage has room for (the planner never puts more tips in a chunk)
  unsigned flags;                    // bit0: R semantics at the root
  long long pat0, pat_end;           // this launch covers patterns [pat0, pat_end) (a segment of the engine's pattern list)
  int part0;                         // first slot of `partials` of this launch
  int parts_total;                   // CTAs of ALL launches of this evaluation: the last one to finish adds the partials up
  unsigned* done_counter;            // zero between evaluations
  double* lnl_out;                   // the evaluation's log-likelihood (weighted sum of the site values)
  const double* rootfreq;            // [4]
  const double* probs;               // [C]
  const double* weights;             // [N]
  double* SR;                        // [N]
  int* rexp;                         // [N]
  double* site_lnl;                  // [N]
  double* partials;                  // [gridDim.x]
};

// (mbarrier / cp.async.bulk helpers: common.cuh)

// explicit shared-space accesses on 32-bit shared addresses (no generic-address LD/ST, no 64-bit pointer arithmetic)
__device__ __forceinline__ double2 lds128(unsigned a) {
  double2 r;
  asm volatile("ld.shared.v2.f64 {%0,%1}, [%2];" : "=d"(r.x), "=d"(r.y) : "r"(a));
  return r;
}
__device__ __forceinline__ void sts128(unsigned a, double x, double y) {
  asm volatile("st.shared.v2.f64 [%2], {%0,%1};" ::"d"(x), "d"(y), "r"(a) : "memory");
}
__device__ __forceinline__ int lds32(unsigned a) {
  int r;
  asm volatile("ld.shared.s32 %0, [%1];" : "=r"(r) : "r"(a));
  return r;
}
__device__ __forceinline__ void sts32(unsigned a, int x) { asm volatile("st.shared.s32 [%1], %0;" ::"r"(x), "r"(a) : "memory"); }
__device__ __forceinline__ unsigned long long lds64u(unsigned a) {
  unsigned long long r;
  asm volatile("ld.shared.u64 %0, [%1];" : "=l"(r) : "r"(a));
  return r;
}

__device__ __forceinline__ unsigned lds_u8(unsigned a) {
  unsigned r;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(r) : "r"(a));
  return r;
}

template <int C_LOG2, int PT, int NW>
struct W4cState {
  static constexpr int C = 1 << C_LOG2;
  static constexpr int NTH = NW * 32;
  static constexpr int PPC = (NW >> C_LOG2) * 32 * PT;
  double v[PT][4], w[PT][4];   // current CLV rows / register slot
  int E[PT], EW[PT];
  unsigned ca;                 // shared address of this thread's code byte of the next tip (pattern j: + 32 j)
  unsigned sp;                 // shared address of the next table block of the current chunk (warp-uniform)
  int tip_off;                 // c * ncodes * 32 bytes
  int tip_block;               // C * ncodes * 32 bytes
  int wide_W;                  // codes of a wide tip (ncodes^2)
  int c;
  unsigned stA, stB, ste;      // shared addresses of the stack planes, already offset by this thread's lane

  // a tip's rows; a wide tip (wide: warp-uniform) also adds its rows' exponents to e
  __device__ __forceinline__ void term_tip(double (&t)[PT][4], int (&e)[PT], bool wide) {
    const unsigned tb = sp + (wide ? (unsigned)(c * wide_W) << 5 : (unsigned)tip_off);
    unsigned code[PT];
#pragma unroll
    for (int j = 0; j < PT; ++j) code[j] = lds_u8(ca + 32 * j);
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      const double2 a = lds128(tb + (code[j] << 5));
      const double2 b = lds128(tb + (code[j] << 5) + 16);
      t[j][0] = a.x; t[j][1] = a.y; t[j][2] = b.x; t[j][3] = b.y;
    }
    if (wide) {
      const unsigned te = sp + ((unsigned)(C * wide_W) << 5) + ((unsigned)(c * wide_W) << 2);
#pragma unroll
      for (int j = 0; j < PT; ++j) e[j] += lds32(te + (code[j] << 2));
    }
    ca += PPC;
    sp += wide ? (unsigned)w4c_wide_block_bytes(C, wide_W) : (unsigned)tip_block;
  }
  // t = P . l, l from: the current rows (W4C_REG), the register slot (W4C_RSL) or a shared-memory slot (W4C_SLOT)
  template <int SRC>
  __device__ __forceinline__ void term_internal(int slot, double (&t)[PT][4], int (&e)[PT]) {
    const unsigned Pm = sp + (c << 7);
    sp += 128 * C;
    double l[PT][4];
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      if (SRC == W4C_SLOT) {
        const unsigned k = (unsigned)((slot * PT + j) * NTH);
        const double2 a = lds128(stA + k * 16), b = lds128(stB + k * 16);
        l[j][0] = a.x; l[j][1] = a.y; l[j][2] = b.x; l[j][3] = b.y;
        e[j] += lds32(ste + k * 4);
      } else if (SRC == W4C_RSL) {
        l[j][0] = w[j][0]; l[j][1] = w[j][1]; l[j][2] = w[j][2]; l[j][3] = w[j][3];
        e[j] += EW[j];
      } else {
        l[j][0] = v[j][0]; l[j][1] = v[j][1]; l[j][2] = v[j][2]; l[j][3] = v[j][3];
        e[j] += E[j];
      }
    }
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const double2 p01 = lds128(Pm + 32 * x);        // warp-uniform address: broadcast
      const double2 p23 = lds128(Pm + 32 * x + 16);
#pragma unroll
      for (int j = 0; j < PT; ++j) t[j][x] = w4c_dot(p01.x, p01.y, p23.x, p23.y, l[j][0], l[j][1], l[j][2], l[j][3]);
    }
  }
  // rescale per row, then store to v (or to the register slot)
  template <bool DSTW>
  __device__ __forceinline__ void commit(double (&a)[PT][4], int (&e)[PT]) {
    int m[PT];
    int mmin = 0x7fffffff;
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      m[j] = w4c_max_hi(a[j]);
      mmin = min(mmin, m[j]);
    }
    if (mmin < kScaleThresholdHi) {  // rare: some row of this thread is small (or identically zero)
#pragma unroll
      for (int j = 0; j < PT; ++j) w4c_rescale(a[j], m[j], e[j]);
    }
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      if (DSTW) {
        w[j][0] = a[j][0]; w[j][1] = a[j][1]; w[j][2] = a[j][2]; w[j][3] = a[j][3];
        EW[j] = e[j];
      } else {
        v[j][0] = a[j][0]; v[j][1] = a[j][1]; v[j][2] = a[j][2]; v[j][3] = a[j][3];
        E[j] = e[j];
      }
    }
  }
  // the four binary shapes.  IEEE multiplication commutes exactly, so (tip, reg) and (reg, tip) -- and the two orders of a
  // join -- are one handler each; the host lays the op's table blocks out in the handler's order (tip block first / the
  // stacked operand's P first).
  template <bool DSTW>
  __device__ __forceinline__ void op_tt(bool wa, bool wb) {
    double ta[PT][4], tb[PT][4];
    int e[PT];
#pragma unroll
    for (int j = 0; j < PT; ++j) e[j] = 0;
    term_tip(ta, e, wa);
    term_tip(tb, e, wb);
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      ta[j][0] *= tb[j][0]; ta[j][1] *= tb[j][1]; ta[j][2] *= tb[j][2]; ta[j][3] *= tb[j][3];
    }
    commit<DSTW>(ta, e);
  }
  template <bool DSTW>
  __device__ __forceinline__ void op_ts(bool wa) {
    double ta[PT][4], tb[PT][4];
    int e[PT];
#pragma unroll
    for (int j = 0; j < PT; ++j) e[j] = 0;
    term_tip(ta, e, wa);
    term_internal<W4C_REG>(0, tb, e);
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      ta[j][0] *= tb[j][0]; ta[j][1] *= tb[j][1]; ta[j][2] *= tb[j][2]; ta[j][3] *= tb[j][3];
    }
    commit<DSTW>(ta, e);
  }
  template <int SRC, bool DSTW>
  __device__ __forceinline__ void op_join(int slot) {
    double ta[PT][4], tb[PT][4];
    int e[PT];
#pragma unroll
    for (int j = 0; j < PT; ++j) e[j] = 0;
    term_internal<SRC>(slot, ta, e);
    term_internal<W4C_REG>(0, tb, e);
#pragma unroll
    for (int j = 0; j < PT; ++j) {
      ta[j][0] *= tb[j][0]; ta[j][1] *= tb[j][1]; ta[j][2] *= tb[j][2]; ta[j][3] *= tb[j][3];
    }
    commit<DSTW>(ta, e);
  }
  // any number of sons in the reference's son order; toks: 2 bits per child (kind), slots: 6 bits per W4C_SLOT child in order
  // of appearance
  __device__ __forceinline__ void op_generic(int nchild, unsigned toks, unsigned slots, bool dstw) {
    double a[PT][4];
    int e[PT];
#pragma unroll
    for (int j = 0; j < PT; ++j) e[j] = 0;
#pragma unroll 1
    for (int ch = 0; ch < nchild; ++ch, toks >>= 2) {
      const int kind = (int)toks & 3;
      double t[PT][4];
      if (kind == W4C_TIP) term_tip(t, e, false);
      else if (kind == W4C_SLOT) { term_internal<W4C_SLOT>((int)slots & 63, t, e); slots >>= 6; }
      else if (kind == W4C_RSL) term_internal<W4C_RSL>(0, t, e);
      else term_internal<W4C_REG>(0, t, e);
#pragma unroll
      for (int j = 0; j < PT; ++j) {
        if (ch == 0) {
          a[j][0] = t[j][0]; a[j][1] = t[j][1]; a[j][2] = t[j][2]; a[j][3] = t[j][3];
        } else {
          a[j][0] *= t[j][0]; a[j][1] *= t[j][1]; a[j][2] *= t[j][2]; a[j][3] *= t[j][3];
        }
      }
    }
    if (dstw) commit<true>(a, e);
    else commit<false>(a, e);
  }
};

// bytes of one ring stage: the table chunk + the tip-code rows of the chunk's tips
__host__ __device__ inline size_t walk4c_stage_bytes(int CH, int C, int PT, int NW, int max_tips) {
  return (size_t)CH + (size_t)max_tips * (NW / C) * 32 * PT;
}
// dynamic shared memory of one CTA: the ring (re-used by the root reduction, which needs 12 bytes per pattern and class), the
// stack planes, the barriers
__host__ __device__ inline size_t walk4c_smem_bytes(int CH, int nslots, int C, int PT, int NW, int max_tips) {
  size_t ring = (size_t)kW4cStages * walk4c_stage_bytes(CH, C, PT, NW, max_tips);
  const size_t root = (size_t)PT * NW * 32 * 12;
  if (ring < root) ring = root;
  return ring + (size_t)(nslots > 0 ? nslots : 0) * PT * NW * 32 * 36 + 128;
}
__host__ __device__ constexpr int walk4c_min_ctas(int PT, int NW) { return NW == 8 ? (PT <= 2 ? 2 : 1) : (PT <= 3 ? 3 : 2); }

template <int C_LOG2, int PT, int NW>
__global__ void __launch_bounds__(NW * 32, walk4c_min_ctas(PT, NW))
walk4c_kernel(const __grid_constant__ Walk4cParams prm, const __grid_constant__ W4cProgram prog) {
  constexpr int C = 1 << C_LOG2;
  constexpr int NTH = NW * 32;
  constexpr int G = NW >> C_LOG2;          // pattern groups (of 32 * PT patterns) per CTA
  constexpr int PPC = G * 32 * PT;         // patterns per CTA
  extern __shared__ __align__(32) unsigned char smem_raw[];
  __shared__ double red[32];

  const int CH = prm.CH;
  const unsigned SB = (unsigned)CH + (unsigned)prm.max_tips * PPC;   // stage bytes
  unsigned char* ring = smem_raw;
  const unsigned ring_s = smem_u32(smem_raw);
  size_t ring_bytes = (size_t)kW4cStages * SB;
  if (ring_bytes < (size_t)PT * NTH * 12) ring_bytes = (size_t)PT * NTH * 12;
  unsigned char* q0 = smem_raw + ring_bytes;
  const size_t plane = (size_t)(prm.nslots > 0 ? prm.nslots : 0) * PT * NTH;
  W4cState<C_LOG2, PT, NW> s;
  s.stA = smem_u32(q0) + threadIdx.x * 16;
  s.stB = smem_u32(q0 + plane * 16) + threadIdx.x * 16;
  s.ste = smem_u32(q0 + plane * 32) + threadIdx.x * 4;
  double* rsum = reinterpret_cast<double*>(smem_raw);                 // [C][PPC] class terms of the root reduction: the ring's
  int* rexpn = reinterpret_cast<int*>(smem_raw + (size_t)PT * NTH * 8);   // [C][PPC]   memory, free once the walk is over
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(q0 + plane * 36);  // full[], empty[]

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int c = warp & (C - 1), g = warp >> C_LOG2;
  s.c = c;
  s.tip_off = c * prm.ncodes * 32;
  s.tip_block = C * prm.ncodes * 32;
  s.wide_W = prm.wide_codes;
  const unsigned my_code_off = (unsigned)(g * (32 * PT) + lane);
#pragma unroll
  for (int j = 0; j < PT; ++j) {
    s.v[j][0] = s.v[j][1] = s.v[j][2] = s.v[j][3] = 1.0;
    s.w[j][0] = s.w[j][1] = s.w[j][2] = s.w[j][3] = 1.0;
    s.E[j] = 0;
    s.EW[j] = 0;
  }

  unsigned long long* full = bars;
  unsigned long long* empty = bars + kW4cStages;
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < kW4cStages; ++i) {
      mbar_init(full + i, 1);
      mbar_init(empty + i, NW);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  __syncthreads();
  const int nchunks = prm.nchunks;
  const unsigned char* my_codes = prm.codesC + (size_t)blockIdx.x * prm.ntips * PPC;
  // producer (thread 0): the tables of chunk k and the code rows of its tips, both completing on full[stage]
  auto issue = [&](int k, int st) {
    const unsigned rec = prog.chunk[k];
    const unsigned tip0 = rec & 0xffffu, ntc = (rec >> 16) & 31u;
    mbar_expect_tx(full + st, (unsigned)CH + ntc * PPC);
    bulk_g2s(ring + (size_t)st * SB, prm.stream + (size_t)k * CH, (unsigned)CH, full + st);
    if (ntc) bulk_g2s(ring + (size_t)st * SB + CH, my_codes + (size_t)tip0 * PPC, ntc * PPC, full + st);
  };
  if (tid == 0)
    for (int k = 0; k < kW4cStages && k < nchunks; ++k) issue(k, k);

  int stage = 0;
  unsigned phase = 0;
  int opi = 0;   // next descriptor
  for (int k = 0; k < nchunks; ++k) {
    const int n_ops = (int)(prog.chunk[k] >> 21) & 31;
    mbar_wait(full + stage, phase);
    s.sp = ring_s + (unsigned)stage * SB;
    s.ca = s.sp + (unsigned)CH + my_code_off;
    for (int o = 0; o < n_ops; ++o) {
      const uint2 dd = prog.desc[opi + o];
      const unsigned d = dd.x;
      const bool wa = d & W4C_WA, wb = d & W4C_WB;
      if (!(d & W4C_DSTW)) {
        if (d & W4C_TS) s.template op_ts<false>(wa);
        else if (d & W4C_TT) s.template op_tt<false>(wa, wb);
        else if (d & W4C_JW) s.template op_join<W4C_RSL, false>(0);
        else if (d & W4C_JS) s.template op_join<W4C_SLOT, false>((int)(d >> 16) & 63);
        else s.op_generic((int)(d >> 24) & 0xf, dd.y & 0xfffu, dd.y >> 12, false);
      } else {
        if (d & W4C_TS) s.template op_ts<true>(wa);
        else if (d & W4C_TT) s.template op_tt<true>(wa, wb);
        else if (d & W4C_JW) s.template op_join<W4C_RSL, true>(0);
        else if (d & W4C_JS) s.template op_join<W4C_SLOT, true>((int)(d >> 16) & 63);
        else s.op_generic((int)(d >> 24) & 0xf, dd.y & 0xfffu, dd.y >> 12, true);
      }
      if (d & 0x4000u) {                            // bit 14: the result is also pushed to a shared-memory slot
        const int dst = (int)(d >> 8) & 0x3f;
#pragma unroll
        for (int j = 0; j < PT; ++j) {
          const unsigned kk = (unsigned)((dst * PT + j) * NTH);
          sts128(s.stA + kk * 16, s.v[j][0], s.v[j][1]);
          sts128(s.stB + kk * 16, s.v[j][2], s.v[j][3]);
          sts32(s.ste + kk * 4, s.E[j]);
        }
      }
    }
    // this warp is done with the stage; the producer refills the stage of the PREVIOUS chunk (one chunk of slack between
    // the slowest warp and the producer's warp), so chunks k+1 .. k+kW4cStages-2 are always loaded or in flight
    __syncwarp();
    if (lane == 0) mbar_arrive(empty + stage);
    if (tid == 0 && k >= 1 && k - 1 + kW4cStages < nchunks) {
      const int ps = stage == 0 ? kW4cStages - 1 : stage - 1;          // stage of chunk k-1
      const unsigned pph = stage == 0 ? phase ^ 1u : phase;             // its phase
      mbar_wait(empty + ps, pph);
      issue(k - 1 + kW4cStages, ps);
    }
    opi += n_ops;
    if (++stage == kW4cStages) { stage = 0; phase ^= 1u; }
  }

  // ---- root reduction: L_i = sum_c p_c 2^-(E_c - Emin) sum_x pi_x CLV_root[i][c][x] (association as in walk4_kernel) ----
  __syncthreads();   // every warp has read its last chunk: the ring is free
  const bool rsem = prm.flags & 1u;
  const double f0 = prm.rootfreq[0], f1 = prm.rootfreq[1], f2 = prm.rootfreq[2], f3 = prm.rootfreq[3];
#pragma unroll
  for (int j = 0; j < PT; ++j) {
    const double t0 = s.v[j][0] * f0, t1 = s.v[j][1] * f1, t2 = s.v[j][2] * f2, t3 = s.v[j][3] * f3;
    double sum;
    if (rsem) sum = (t0 > 0 ? t0 : 0.0) + (t1 > 0 ? t1 : 0.0) + (t2 > 0 ? t2 : 0.0) + (t3 > 0 ? t3 : 0.0);
    else sum = ((t0 + t1) + t2) + t3;
    const int lp = g * (32 * PT) + 32 * j + lane;   // pattern index inside the CTA
    rsum[c * PPC + lp] = sum;
    rexpn[c * PPC + lp] = s.E[j];
  }
  __syncthreads();
  double contrib = 0.0;
  for (int lp = tid; lp < PPC; lp += NTH) {
    const long long pat = prm.pat0 + (long long)blockIdx.x * PPC + lp;
    if (pat >= prm.pat_end) continue;
    int Emin = rexpn[lp];
#pragma unroll
    for (int cc = 1; cc < C; ++cc) Emin = min(Emin, rexpn[cc * PPC + lp]);
    double Lc[C];
#pragma unroll
    for (int cc = 0; cc < C; ++cc) {
      double L = rsum[cc * PPC + lp] * align_factor(rexpn[cc * PPC + lp] - Emin) * prm.probs[cc];
      if (rsem && !(L > 0)) L = 0.0;
      Lc[cc] = L;
    }
#pragma unroll
    for (int off = 1; off < C; off <<= 1)      // the xor-butterfly order of walk4_kernel, as seen by class 0
#pragma unroll
      for (int cc = 0; cc < C; cc += 2 * off) Lc[cc] += Lc[cc + off];
    double L = Lc[0];
    if (!rsem && L < 0) L = 0.0;
    const double lnl = log(L) - (double)Emin * kLn2;
    prm.SR[pat] = L;
    prm.rexp[pat] = Emin;
    prm.site_lnl[pat] = lnl;
    contrib += prm.weights[pat] * lnl;
  }
  const double bs = block_sum(contrib, red);
  // the CTA that finishes last (over every launch of the evaluation) sums the per-CTA partials in index order: the same
  // fixed-shape, deterministic reduction a separate finalize launch would do, without the launch
  __shared__ bool is_last;
  if (tid == 0) {
    prm.partials[prm.part0 + blockIdx.x] = bs;
    __threadfence();
    const unsigned ticket = atomicAdd(prm.done_counter, 1u);
    is_last = ticket == (unsigned)prm.parts_total - 1u;
  }
  __syncthreads();
  if (is_last) {
    __threadfence();
    double acc = 0.0;
    for (int i = tid; i < prm.parts_total; i += NTH) acc += __ldcg(prm.partials + i);
    const double tot = block_sum(acc, red);
    if (tid == 0) {
      *prm.lnl_out = tot;
      *prm.done_counter = 0u;
    }
  }
}

// codes [nl][N] (leaf-slot major) -> codesC [cta][tip in consumption order][PPC]: the rows a CTA stages with its chunks
// (of one segment [pat0, pat_end) of the pattern list, walked by CTAs of PPC patterns).  A tip entry is {leaf slot, -1}; a
// folded cherry's is {leaf slot of son 0, leaf slot of son 1}, whose row is the mixed-radix code code_0 * ncodes + code_1.
__global__ void pack_codesC_kernel(const unsigned char* codes, const int2* tip_order, int ntips, int ncodes, long long N,
                                   long long pat0, long long pat_end, int PPC, unsigned char* codesC) {
  const size_t cta = blockIdx.x;
  for (int i = threadIdx.x; i < ntips * PPC; i += blockDim.x) {
    const int k = i / PPC, p = i - k * PPC;
    const long long pat = pat0 + (long long)cta * PPC + p;
    unsigned v = 0;
    if (pat < pat_end) {
      const int2 t = tip_order[k];
      v = codes[(size_t)t.x * N + pat];
      if (t.y >= 0) v = v * (unsigned)ncodes + codes[(size_t)t.y * N + pat];
    }
    codesC[(cta * ntips + k) * PPC + p] = (unsigned char)v;
  }
}

// table blocks of the chunked stream: one CTA per child block
struct Pack4cBlock {
  int kind;       // W4C_TIP, W4C_CHERRY or internal
  int pnode;      // node whose branch carries the child
  int son0, son1; // W4C_CHERRY: the cherry's tips, son order
  long long off;  // BYTE offset of the block in the chunked stream
};

// [class][code][x]: P . (code's tip vector), one tip table
__device__ __forceinline__ void w4c_tip_block(const double* Pn, const double* code_table, int C, int ncodes, double* out) {
  for (int e = threadIdx.x; e < ncodes * C * 4; e += blockDim.x) {
    const int x = e & 3, code = (e >> 2) % ncodes, c = (e >> 2) / ncodes;
    const double* tv = code_table + code * 4;
    const double* pr = Pn + c * 16 + x * 4;
    out[e] = w4c_dot(pr[0], pr[1], pr[2], pr[3], tv[0], tv[1], tv[2], tv[3]);
  }
}
// the wide-tip block of a folded cherry (layout: w4c_wide_block_bytes).  Per (class, code pair) row the steps of the walk's
// op_tt on the two tips -- tip terms, product, rescale -- and then term_internal of the father's contraction with the
// cherry's branch P: the row the father would have read, with the exponent it would have added.
__device__ __forceinline__ void w4c_cherry_block(const double* Pa, const double* Pb, const double* Pn, const double* code_table,
                                                 int C, int ncodes, unsigned char* out) {
  const int W = ncodes * ncodes;
  double* rows = reinterpret_cast<double*>(out);
  int* exps = reinterpret_cast<int*>(out + (size_t)C * W * 32);
  for (int r = threadIdx.x; r < C * W; r += blockDim.x) {
    const int c = r / W, code = r - c * W;
    const double* ta = code_table + (code / ncodes) * 4;
    const double* tb = code_table + (code % ncodes) * 4;
    double a[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const double* pa = Pa + c * 16 + x * 4;
      const double* pb = Pb + c * 16 + x * 4;
      a[x] = w4c_dot(pa[0], pa[1], pa[2], pa[3], ta[0], ta[1], ta[2], ta[3]) *
             w4c_dot(pb[0], pb[1], pb[2], pb[3], tb[0], tb[1], tb[2], tb[3]);
    }
    int e = 0;
    w4c_rescale(a, w4c_max_hi(a), e);
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const double* pn = Pn + c * 16 + x * 4;
      rows[(size_t)r * 4 + x] = w4c_dot(pn[0], pn[1], pn[2], pn[3], a[0], a[1], a[2], a[3]);
    }
    exps[r] = e;
  }
}

__global__ void pack_stream4c_kernel(const Pack4cBlock* blocks, const double* P /*[nn][C][4][4]*/, const double* code_table,
                                     int C, int ncodes, unsigned char* stream) {
  const Pack4cBlock b = blocks[blockIdx.x];
  const double* Pn = P + (size_t)b.pnode * C * 16;
  double* out = reinterpret_cast<double*>(stream + b.off);
  if (b.kind == W4C_TIP) {
    w4c_tip_block(Pn, code_table, C, ncodes, out);
  } else if (b.kind == W4C_CHERRY) {
    w4c_cherry_block(P + (size_t)b.son0 * C * 16, P + (size_t)b.son1 * C * 16, Pn, code_table, C, ncodes, stream + b.off);
  } else {                   // [class][x][y] = the reference's pxy_ order
    for (int e = threadIdx.x; e < C * 16; e += blockDim.x) out[e] = Pn[e];
  }
}

// K1 + K2b fused for the DNA walk (S = 4, real spectra, value only): the CTA of a child block builds the branch's
// P(t) = V exp(L r_c t) V^-1 for every class -- the arithmetic of pt_eigen_kernel (pt_kernels.cuh), term by term, so the tables are
// bit-identical -- writes it to the P table (accessors read it there) and lays out its stream block.  One launch instead of two.
// A cherry block builds the P of its three branches (both tips' and the cherry's own).
struct PtPack4cParams {
  const Pack4cBlock* blocks;
  const ModelDev* models;
  const int* branch_model;   // [nn] of this point
  const double* brlen;       // [nn] of this point
  const double* rates;       // [C]
  const double* code_table;
  int C, ncodes;
  double* P;                 // [nn][C][4][4] of this point
  unsigned char* stream;
};
__device__ __forceinline__ void pt4c_branch(const PtPack4cParams& p, int node, double* Ps) {
  const ModelDev md = p.models[p.branch_model[node]];
  const int C = p.C;
  for (int e = threadIdx.x; e < C * 16; e += blockDim.x) {
    const int c = e >> 4, x = (e >> 2) & 3, y = e & 3;
    const double l = md.rate * (p.brlen[node] * p.rates[c]);
    double a0 = 0.0;
#pragma unroll
    for (int k = 0; k < 4; ++k) a0 = fma(md.V[x * 4 + k] * md.Vinv[k * 4 + y], exp(md.re[k] * l), a0);
    Ps[e] = a0;
    p.P[(size_t)node * C * 16 + e] = a0;
  }
}
__global__ void pt_pack4c_kernel(PtPack4cParams p) {
  __shared__ double Ps[3][8 * 16];
  const Pack4cBlock b = p.blocks[blockIdx.x];
  const int C = p.C;
  pt4c_branch(p, b.pnode, Ps[0]);
  if (b.kind == W4C_CHERRY) {
    pt4c_branch(p, b.son0, Ps[1]);
    pt4c_branch(p, b.son1, Ps[2]);
  }
  __syncthreads();
  double* out = reinterpret_cast<double*>(p.stream + b.off);
  if (b.kind == W4C_TIP) {
    w4c_tip_block(Ps[0], p.code_table, C, p.ncodes, out);
  } else if (b.kind == W4C_CHERRY) {
    w4c_cherry_block(Ps[1], Ps[2], Ps[0], p.code_table, C, p.ncodes, p.stream + b.off);
  } else {
    for (int e = threadIdx.x; e < C * 16; e += blockDim.x) out[e] = Ps[0][e];
  }
}

}  // namespace bppgpu
