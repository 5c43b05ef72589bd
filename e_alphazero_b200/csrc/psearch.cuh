// psearch.cuh -- the PERSISTENT search kernel for one-hot (DeepSea) observations and the per-cell network table it reads (included by
// search.cu).
//
// Every network evaluation of a DeepSea search has a one-hot observation with a single cell (deepsea_obs_index), so the three head
// outputs the search needs -- value, UBE (novelty and clamp included) and the policy head's logits -- are a pure function of (model,
// cell).  ds_output_table_kernel computes them for all N x N cells once per model, beside the other parameter-derived tables (h1 rows,
// ds_seen; skipped under EAZ_FLAG_REUSE_PREPARED), and the search kernel reads one float4 per leaf from that table instead of evaluating
// the network per simulation (at C2: ~2.1 M evaluations of 900 distinct inputs per model).
//
// ds_output_table_kernel: one CTA per (head, 128-cell tile).  8 gather warps copy the pre-activated fp16 hi/lo layer-1 rows
// (mlp_gather.cu: h1 table) of the tile's cells straight into tensor memory, one warp streams the W2 chunk images (K = 16 chunks) with
// 1-D bulk async copies, one elected thread issues tcgen05.mma kind::f16 (M=128, N=256, K=16, 3 split-precision products per chunk)
// into a TMEM accumulator, and 16 warps run layer 3 (<= 2 outputs) on the CUDA cores straight out of TMEM.
//
// ds_search_kernel: one CTA owns kSlots trees for the WHOLE search (all num_simulations simulations, the loop the reference runs as one
// compiled lax.fori_loop: /root/reference/src/selfplay.py:107-117,148).  Nothing is re-launched, re-allocated or re-staged between
// simulations: 16 tree warps (two trees per warp, 16 lanes each -- the mapping of tree_step2_kernel) keep, per tree and for the whole
// search, the cached selection and the compact env state of EVERY node in shared memory (the pointer-chase descent never leaves the
// SM), plus a staging area with the node / edge records of the current path.  Per simulation a tree warp runs: expand (with the leaf's
// table entry) + backward + action refresh (tree_step.cuh: staged2_*, the staged step of tree_step2_kernel) -> descent over the cached
// selections -> cp.async copies of the new path's records into the staging area -> DeepSea transition -> load of the new leaf's table
// entry -> wait for the copies and finish the staging.  Trees that cannot be staged (path longer than kNodes - 1, re-expanded leaf
// under a max_depth cut-off) take tree_step_direct for that simulation and re-synchronise their shared-memory caches.
//
// The tree itself (node / edge records, states) still lives in the caller's workspace in HBM/L2 -- it is the search's OUTPUT
// (finalize / export read it) and the source of the staging copies -- but the per-simulation critical path touches it only with
// fire-and-forget stores and one round trip of staging copies.  Measured at C2 (B200, 1000 W): 6.0 us mean period per simulation and
// warp -- refresh 2.44, descent incl. the copy issue and transition 1.67, backward 1.03, staging 0.63, expand 0.25 us
// (profiles/r5_trace_psearch_c2.txt).
#pragma once
#include "umma.cuh"

namespace eaz {
namespace ps {
using namespace umma;

constexpr int kHeads = 3;   // value, UBE, policy (one table CTA each)
constexpr int kH = 256;
constexpr int kCK = 16;               // K (halves) per chunk = one tcgen05.mma kind::f16 K-step
constexpr int kChunks = kH / kCK;     // 16 per evaluation
constexpr int kRows = 128;            // table cells per CTA = MMA M = TMEM lanes
// W2 chunk ring of the table kernel (the A operand lives in tensor memory: no A ring)
constexpr int kStages = 5;
constexpr int kBHalf = kH * kCK * 2;     // 8 KB: hi or lo tile of a W2 chunk
constexpr int kBStage = 2 * kBHalf;
// tensor memory (512 columns x 128 lanes): D = relu-input accumulator [0, 256); A operand of the whole K = 256, written by the gather
// warps with tcgen05.st and read by tcgen05.mma straight from TMEM: hi halves [256, 384), lo halves [384, 512), 8 columns per chunk
constexpr int kTmemCols = 512, kTmemAhi = 256, kTmemAlo = 384, kAColsPerChunk = kCK / 2;
constexpr int kSBO = (kCK * 2 / 16) * kCoreBytes;  // 256 B between 8-row groups
constexpr int kL3Warps = 16, kGWarps = 8;          // layer 3: 4 TMEM lane quarters x 4 groups of 64 columns; warps 0..7 gather first
constexpr int kWarpMma = kL3Warps, kWarpCopy = kL3Warps + 1;
constexpr int kTableThreads = (kL3Warps + 2) * 32;
constexpr int kBarL3 = 1;  // named barrier: layer-3 partial sums
// (activation scale kActScale = 16: mlp.cuh; the W2 images carry a per-matrix power-of-two scale: TableArgs::wscale)

struct TableShared {
  uint64_t full_a[kChunks];  // chunk c of the A operand is in tensor memory (4 arrivals: one per 32-row quarter)
  uint64_t full_b[kStages], empty[kStages];
  uint64_t acc_done;  // the MMAs are complete (tcgen05.commit)
  uint32_t tmem_base, pad;
  alignas(16) float b2[kH];
  alignas(16) float w3t[2][kH];         // layer-3 weights, output-major
  alignas(16) float part[3][kRows][2];  // layer-3 partial sums of column groups 1..3
};
constexpr size_t kTableSmem = 1024 + (size_t)kStages * kBStage + sizeof(TableShared);

struct TableArgs {
  // per head (blockIdx.y): the W2 chunk images (K = 16 chunks), the layer-1 row table, b2, W3, b3
  const uint8_t* w2img[kHeads];
  const uint8_t* h1[kHeads];
  const float* b2[kHeads];
  const float* w3[kHeads];
  const float* b3[kHeads];
  int nout[kHeads];
  int head_id[kHeads];  // EAZ_HEAD_*
  const float* wscale;  // [4][3] power-of-two scales of the weight images (tile_weights.cu)
  const uint8_t* ds_seen;
  float max_u, novelty_scale;
  int cells;   // N x N
  float4* out;  // [cells] {value, ube, logit 0, logit 1}
};

// ---- the network of one head for 128 rows, split by role

// weight-copy warp, one lane: the W2 chunk ring (kChunks chunks through kStages stages)
__device__ __forceinline__ void w2_ring_copy(const uint8_t* img, uint8_t* sB, TableShared* sh) {
#pragma unroll 1
  for (int g = 0; g < kChunks; ++g) {
    const int s = g % kStages;
    if (g >= kStages) mbar_wait(&sh->empty[s], ((g / kStages) & 1) ^ 1);
    mbar_arrive_expect_tx(&sh->full_b[s], (uint32_t)kBStage);
    bulk_g2s(sB + s * kBStage, img + (size_t)g * kBStage, kBStage, &sh->full_b[s]);
  }
}

// MMA-issue warp: the whole warp runs the loop with warp-uniform values and ONE ELECTED lane issues (inside an `if (lane == 0)` region
// the compiler treats the descriptors as per-thread values and wraps every tcgen05.mma in an ELECT / R2UR.BROADCAST loop, ~100 cycles
// per instruction, measured: 1000 cycles per 3-MMA chunk against 384 cycles of tensor work).
__device__ __forceinline__ void mma_issue(const uint8_t* sB, TableShared* sh) {
  const uint32_t tmem = sh->tmem_base;
  const uint32_t desc_hi = (uint32_t)(kSBO >> 4) | (1u << 14);  // SBO [32,46) + version=1 [46,48)
  const uint32_t lbo_bits = (uint32_t)(kCoreBytes >> 4) << 16;  // LBO [16,30)
  auto mk = [&](uint32_t lo) { return ((uint64_t)desc_hi << 32) | (uint64_t)lo; };
  const uint32_t idesc = idesc_f16(kRows, kH);
  const uint32_t b_base = ((smem_u32(sB) & 0x3FFFFu) >> 4) | lbo_bits;
#pragma unroll 1
  for (int c = 0; c < kChunks; ++c) {
    const int s = c % kStages, ph = (c / kStages) & 1;
    mbar_wait(&sh->full_a[c], 0);  // (all 32 lanes: uniform control flow)
    mbar_wait(&sh->full_b[s], ph);
    tc_fence_after();
    const uint32_t bl = b_base + (uint32_t)((s * kBStage) >> 4);
    const uint32_t a_hi = tmem + (uint32_t)(kTmemAhi + c * kAColsPerChunk), a_lo = tmem + (uint32_t)(kTmemAlo + c * kAColsPerChunk);
    if (elect_one()) {
      mma_f16_ts(tmem, a_hi, mk(bl), idesc, c != 0);
      mma_f16_ts(tmem, a_hi, mk(bl + (kBHalf >> 4)), idesc, 1);
      mma_f16_ts(tmem, a_lo, mk(bl), idesc, 1);
      mma_commit(&sh->empty[s]);
      if (c == kChunks - 1) mma_commit(&sh->acc_done);
    }
    __syncwarp();
  }
}

// gather warp gw (0..7): layer 1 = copy of the row's h1 table row into TENSOR MEMORY.  The A operand never touches shared memory:
// thread = row (TMEM lane), a chunk of a row is 32 bytes of hi and 32 bytes of lo halves = 2 x 8 tensor-memory columns, written with
// tcgen05.st and consumed by tcgen05.mma with A in TMEM.  (With A in shared memory a chunk moved 60 KB through the SM's shared-memory
// port -- 36 KB of operand reads for the three split-precision products, 24 KB of ring writes -- i.e. >= 470 cycles against 384 cycles
// of tensor work; measured 630.)  The whole K = 256 of a row fits beside the accumulator, so there is no A ring.  Warp gw serves the 32
// rows of TMEM quarter gw % 4 (= warp id % 4, the quarter tcgen05.st may address) and the chunks of parity gw / 4.
__device__ __forceinline__ void gather_rows(const uint8_t* table, int cell, int gw, int lane, TableShared* sh) {
  const int q = gw & 3, half = gw >> 2;
  const uint32_t tq = sh->tmem_base + ((uint32_t)(32 * q) << 16);
  const uint4* const src = reinterpret_cast<const uint4*>(table + (size_t)cell * (4 * kH));  // [hi 512 B | lo 512 B]
#pragma unroll 1
  for (int k = 0; k < kChunks / 2; ++k) {
    const int c = 2 * k + half;
    const uint4 v0 = __ldg(src + 2 * c), v1 = __ldg(src + 2 * c + 1);
    const uint4 v2 = __ldg(src + 2 * c + (2 * kH) / 16), v3 = __ldg(src + 2 * c + (2 * kH) / 16 + 1);
    tmem_st8(tq + (uint32_t)(kTmemAhi + c * kAColsPerChunk), v0, v1);
    tmem_st8(tq + (uint32_t)(kTmemAlo + c * kAColsPerChunk), v2, v3);
    tmem_st_wait();
    tc_fence_before();
    __syncwarp();
    if (lane == 0) mbar_arrive(&sh->full_a[c]);
  }
}

// layer-3 warp w (0..15): y = relu(D + b2) @ W3 for the 32 rows of TMEM quarter w % 4 and the 64 accumulator columns of group w / 4.
// Group 0 then adds the partials of groups 1, 2, 3 in that order; returns true (with the row's y0, y1, b3 not yet added) in group 0.
__device__ __forceinline__ bool layer3(TableShared* sh, int w, int lane, int nout, float unscale, float& y0, float& y1) {
  const int q = w & 3, cg = w >> 2;
  const int row = 32 * q + lane;
  const uint32_t taddr = sh->tmem_base + ((uint32_t)(32 * q) << 16) + (uint32_t)(64 * cg);
  y0 = 0.0f;
  y1 = 0.0f;
  uint32_t ra[16], rb[16];
  auto consume16 = [&](const uint32_t (&r)[16], int k0) {
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      const float4 bq = *reinterpret_cast<const float4*>(&sh->b2[k0 + 4 * x]);
      const float h0 = fmaxf(__fmaf_rn(__uint_as_float(r[4 * x + 0]), unscale, bq.x), 0.0f);
      const float h1 = fmaxf(__fmaf_rn(__uint_as_float(r[4 * x + 1]), unscale, bq.y), 0.0f);
      const float h2 = fmaxf(__fmaf_rn(__uint_as_float(r[4 * x + 2]), unscale, bq.z), 0.0f);
      const float h3 = fmaxf(__fmaf_rn(__uint_as_float(r[4 * x + 3]), unscale, bq.w), 0.0f);
      const float4 w0 = *reinterpret_cast<const float4*>(&sh->w3t[0][k0 + 4 * x]);
      y0 = __fmaf_rn(h0, w0.x, y0); y0 = __fmaf_rn(h1, w0.y, y0); y0 = __fmaf_rn(h2, w0.z, y0); y0 = __fmaf_rn(h3, w0.w, y0);
      if (nout > 1) {
        const float4 w1 = *reinterpret_cast<const float4*>(&sh->w3t[1][k0 + 4 * x]);
        y1 = __fmaf_rn(h0, w1.x, y1); y1 = __fmaf_rn(h1, w1.y, y1); y1 = __fmaf_rn(h2, w1.z, y1); y1 = __fmaf_rn(h3, w1.w, y1);
      }
    }
  };
  tmem_ld16(taddr, ra);
  tmem_ld_wait();
  tmem_ld16(taddr + 16, rb);
  consume16(ra, 64 * cg);
  tmem_ld_wait();
  tmem_ld16(taddr + 32, ra);
  consume16(rb, 64 * cg + 16);
  tmem_ld_wait();
  tmem_ld16(taddr + 48, rb);
  consume16(ra, 64 * cg + 32);
  tmem_ld_wait();
  consume16(rb, 64 * cg + 48);
  tc_fence_before();
  if (cg > 0) *reinterpret_cast<float2*>(sh->part[cg - 1][row]) = make_float2(y0, y1);
  asm volatile("bar.sync %0, %1;" ::"r"(kBarL3), "r"(kL3Warps * 32) : "memory");
  if (cg != 0) return false;
#pragma unroll
  for (int pgrp = 0; pgrp < 3; ++pgrp) {
    const float2 o = *reinterpret_cast<const float2*>(sh->part[pgrp][row]);
    y0 = __fadd_rn(y0, o.x);
    y1 = __fadd_rn(y1, o.y);
  }
  return true;
}

// out[cell] = {value, ube, logit 0, logit 1} of every cell; grid (ceil(cells / 128), kHeads), each CTA writes its head's components
__global__ void __launch_bounds__(kTableThreads, 1) ds_output_table_kernel(const __grid_constant__ TableArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sB = smem;
  TableShared* sh = reinterpret_cast<TableShared*>(sB + kStages * kBStage);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int head = blockIdx.y;
  const int nout = a.nout[head];

  if (threadIdx.x == 0) {
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&sh->full_b[s], 1);
      mbar_init(&sh->empty[s], 1);
    }
    for (int c = 0; c < kChunks; ++c) mbar_init(&sh->full_a[c], 4);
    mbar_init(&sh->acc_done, 1);
    fence_mbar_init();
  }
  if (threadIdx.x < kH) {
    const int j = threadIdx.x;
    sh->b2[j] = __ldg(a.b2[head] + j);
    sh->w3t[0][j] = __ldg(a.w3[head] + (size_t)j * nout);
    sh->w3t[1][j] = nout > 1 ? __ldg(a.w3[head] + (size_t)j * nout + 1) : 0.0f;
  }
  if (warp == kWarpMma) {
    tmem_alloc(&sh->tmem_base, kTmemCols);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();

  if (warp == kWarpCopy) {
    if (lane == 0) w2_ring_copy(a.w2img[head], sB, sh);
    __syncwarp();
  } else if (warp == kWarpMma) {
    mma_issue(sB, sh);
  } else {
    const int row = 32 * (warp & 3) + lane;
    const int cell = blockIdx.x * kRows + row;
    const bool live = cell < a.cells;
    if (warp < kGWarps) gather_rows(a.h1[head], live ? cell : 0, warp, lane, sh);
    const int hid = a.head_id[head];
    int seen = 0;  // novelty bit of the row's cell (fully_connected.py:83-90), fetched while the MMAs run
    if (warp >> 2 == 0 && hid == EAZ_HEAD_UBE && live) seen = a.ds_seen[cell];
    mbar_wait_warp(&sh->acc_done, 0);
    tc_fence_after();
    const float unscale = 1.0f / (kActScale * __ldg(a.wscale + 3 * hid + 1));  // exact (powers of two)
    float y0, y1;
    if (layer3(sh, warp, lane, nout, unscale, y0, y1) && live) {
      float* o = reinterpret_cast<float*>(a.out + cell);
      const float b3_0 = __ldg(a.b3[head]);
      if (hid >= EAZ_HEAD_EXPLOIT) {
        o[2] = __fadd_rn(y0, b3_0);
        o[3] = nout > 1 ? __fadd_rn(y1, __ldg(a.b3[head] + 1)) : 0.0f;
      } else {
        const float y = __fadd_rn(y0, b3_0);
        if (hid == EAZ_HEAD_VALUE) {
          o[0] = eaz_tanh(y);
        } else {  // fully_connected.py:92-96
          float u = __fmul_rn(0.5f, __fadd_rn(eaz_tanh(y), 1.0f));
          const float nov = __fmul_rn(seen ? 0.0f : 1.0f, a.novelty_scale);
          u = __fmul_rn(u, a.max_u);
          u = eaz_max(nov, u);
          u = eaz_min(eaz_max(u, 0.0f), a.max_u);
          o[1] = u;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kWarpMma) tmem_dealloc(sh->tmem_base, kTmemCols);
}

// ---- the search kernel
constexpr int kTWarps = 16;          // tree warps per CTA
constexpr int kSlots = 2 * kTWarps;  // trees per CTA
constexpr int kThreads = kTWarps * 32;
// per-tree staging area (uint32 words), sized for kNodes staged nodes (path + leaf).  The edge and back words and the leaf priors
// (misc [8..8+A)) have the layout of tree_step2_kernel's staging area, which the staged step of tree_step.cuh (staged2_*) reads; the
// root words, the other misc words and the 16-bit next words are this kernel's own.
constexpr int kG = 2;                          // lanes per node (A <= 2)
constexpr int kPR = kStaged2Lanes / kG;        // nodes refreshed per round
constexpr int kRounds = 3;
constexpr int kNodes = kRounds * kPR;          // 24
constexpr int kEdgeWords = kRounds * kStaged2LaneWords * kStaged2Lanes;  // 480
constexpr int kRootWords = 4;                  // [a] gumbel + (logit - max logit), [2 + a] invalid flag
constexpr int kMiscWords = 12;                 // [0] considered visit, [1] number of considered actions, [8..8+A) leaf priors
constexpr int kTreeWords = kEdgeWords + kStaged2BackWords + kRootWords + kMiscWords;  // + ncap state words + ncap/2 next words

__host__ __device__ inline int tree_words(int ncap) { return kTreeWords + ncap + ncap / 2; }  // ncap even
constexpr int kAmapMax = 16384;  // the DeepSea action map (N x N bytes) is mirrored in shared memory when it fits (N <= 128)
__host__ __device__ inline int amap_bytes(int size) { return size * size <= kAmapMax ? ((size * size + 15) & ~15) : 0; }
__host__ __device__ inline size_t smem_bytes(int ncap, int size) { return (size_t)kSlots * tree_words(ncap) * 4 + (size_t)amap_bytes(size); }

// A value the compiler may not re-derive (ptxas folds a plain `mov`; a value that went through a warp shuffle -- every lane reads its
// own -- is not recomputable): shared-window addresses for the inner loops.
__device__ __forceinline__ uint32_t opaque_u32(uint32_t v) { return __shfl_sync(0xffffffffu, v, threadIdx.x & 31); }
__device__ __forceinline__ uint32_t lds_u16(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }
// 4-byte global -> shared copy that holds no register until it lands (LDGSTS).  4-byte copies take only the .ca cache operator: the
// read goes through the SM's L1 and L2.
__device__ __forceinline__ void cp_async4(uint32_t dst, const void* src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// Optional timeline of CTA 0 (eaz_debug_set_ps_trace): per simulation `it` and tree warp w, at [(it * kTWarps + w) * 8 + k], globaltimer
// stamps of k = 0 expand done (the leaf's table entry has been used), 1 backward done, 2 refresh done, 3 descent done (the next leaf's
// table load is issued), 4 staging done; k = 5 the longer of the warp's two path lengths (high 32 bits: 1 = DIRECT step).
struct Trace {
  unsigned long long* buf;
  __device__ __forceinline__ void stamp(int it, int w, int k) const {
    if (buf) buf[((size_t)it * kTWarps + w) * 8 + k] = globaltimer_ns();
  }
  __device__ __forceinline__ void path(int it, int w, int L, int direct) const {
    if (buf) buf[((size_t)it * kTWarps + w) * 8 + 5] = (unsigned long long)L | ((unsigned long long)direct << 32);
  }
};

struct Args {
  Tree t;
  SearchParams sp;
  EnvDesc env;
  const float* beta;
  const uint8_t* invalid;
  const float4* ds_out;  // ds_output_table_kernel: {value, ube, logit 0, logit 1} per observation cell
  int ncap;
  unsigned long long* trace;
};

// tree_step_direct for both trees of a tree warp, one after the other with the whole warp (cold path)
__device__ __noinline__ void direct_pair(const Args& a, int sim, int do_backward, int do_select, int b0, int lane) {
#pragma unroll 1
  for (int s2 = 0; s2 < 2; ++s2) {
    const int bb = b0 + s2;
    if (bb < a.t.B) tree_step_direct<kG, 1>(a.t, a.sp, a.env, sim, do_backward, do_select, a.beta ? a.beta[bb] : 0.0f, a.invalid, bb, lane, nullptr);
    __syncwarp();
  }
}

__global__ void __launch_bounds__(kThreads, 1) ds_search_kernel(const __grid_constant__ Args a) {
  extern __shared__ __align__(16) uint32_t tree_smem[];
  uint8_t* const s_amap = reinterpret_cast<uint8_t*>(tree_smem + (size_t)kSlots * tree_words(a.ncap));  // mirror of env.action_map (or unused)
  const int amap_n = a.env.action_map ? amap_bytes(a.env.size) : 0;
  const Tree& t = a.t;
  const SearchParams& sp = a.sp;
  const int tw = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n = sp.n;
  const Trace trc{(a.trace && blockIdx.x == 0) ? a.trace : nullptr};

  if (amap_n)
    for (int i = threadIdx.x; i < a.env.size * a.env.size; i += kThreads) s_amap[i] = a.env.action_map[i];
  __syncthreads();

  // ================================================================ tree warps: two trees each (16 lanes per tree)
  const int hl = lane & (kStaged2Lanes - 1), hbase = lane & kStaged2Lanes, sub = lane >> 4;
  const int slot = 2 * tw + sub;
  const int b0 = blockIdx.x * kSlots + 2 * tw;  // the warp's first tree
  const int b = b0 + sub;
  const bool in_batch = b < t.B;
  const unsigned uB = (unsigned)t.B, uA = (unsigned)t.A, ub = (unsigned)(in_batch ? b : 0);
  const int gl = hl & (kG - 1), glev = hl / kG;
  const bool valid1[1] = {gl < t.A};
  const int ncap = a.ncap;
  uint32_t* const sw = tree_smem + (size_t)slot * tree_words(ncap);
  uint32_t* const s_edge = sw;
  uint32_t* const s_back = sw + kEdgeWords;
  uint32_t* const s_root = s_back + kStaged2BackWords;
  uint32_t* const s_misc = s_root + kRootWords;
  uint32_t* const s_state = s_misc + kMiscWords;
  uint16_t* const s_next = reinterpret_cast<uint16_t*>(s_state + ncap);
  const Staged2Lane w{lane, hl, hbase, gl, glev, valid1[0], in_batch, uB, uA, ub, s_edge, s_back, s_misc};
  const float beta = (in_batch && a.beta) ? a.beta[b] : 0.0f;
  const bool std_backup = (sp.flags & EAZ_FLAG_BACKUP_STD) != 0;
  uint32_t* const st_global = reinterpret_cast<uint32_t*>(t.states);

  // this tree's pending simulation: path length, leaf, reward / terminal flag of the leaf's state, the network outputs of its cell
  int L = 0, leaf = 0;
  float reward = 0.0f;
  float4 net = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
  bool term = false, staged = false;

  // ---- reload everything the persistent state mirrors from the workspace (after a DIRECT step)
  auto resync = [&](int sim) {
    if (in_batch) {
      for (int nd = hl; nd <= sim + 1 && nd < ncap; nd += kStaged2Lanes) {
        s_next[nd] = (uint16_t)pack_next16(t.nodes[(unsigned)nd * uB + ub].pad0);
        s_state[nd] = st_global[(unsigned)nd * uB + ub];
      }
      L = t.path_len[b];
      leaf = t.leaf[b];
      reward = t.reward[b];
      const uint32_t ns = st_global[(unsigned)leaf * uB + ub];
      term = EAZ_DS_TERM(ns) != 0;
      net = __ldg(a.ds_out + deepsea_obs_index(ns, a.env.size));
      for (int lev = hl; lev < L && lev < 32; lev += kStaged2Lanes) {
        const int2 pa = t.path[(unsigned)lev * uB + ub];
        s_back[lev] = (uint32_t)pa.x | ((uint32_t)pa.y << 16);
      }
    }
    __syncwarp();
  };
  // ---- the staging loads of the step for simulation `sim_next`, as cp.async copies straight into the staging slots (no register
  // holds them while they are in flight).  A tree issues all of them at once as soon as its new path is known -- after the descent,
  // ahead of the DeepSea transition and the table load -- and stage() waits for them: one L2 round trip.  (Issued level by level
  // inside the descent instead, their issue cost lengthened the chase by more than it took off the wait; measured at C2 on a B200:
  // descent 1.20 -> 2.21 us, staging 1.31 -> 0.60 us per simulation.)
  // Ordering: the records they read were last written in this simulation's expand, backward and refresh (or its DIRECT step) by
  // lanes of this warp, each phase ending in __syncwarp, which orders those stores before any memory operation the warp's lanes issue
  // after it.  A non-bulk cp.async is a weak read of the generic proxy by the issuing thread, so it sees those stores exactly as the
  // plain loads it replaces did.  The slots it fills were last read by this simulation's backward / refresh, before the same
  // __syncwarp.
  //
  // A tree can be staged when its path fits and its leaf is fresh.  The leaf is fresh exactly when the descent ended on an
  // unexpanded child, which gets the next unused index sim_next (search.py); a descent cut off by max_depth ends on an expanded node
  // (index < sim_next), which takes the DIRECT step.
  auto stageable = [&](int sim_next) { return L + 1 <= kNodes && leaf == sim_next && !(sp.flags & EAZ_FLAG_PUCT); };
  auto issue_staging = [&](int sim_next) {
    if (!in_batch || !stageable(sim_next)) return;
    if (hl == 0) cp_async4(smem_u32(s_misc), t.table + (s_misc[1] * sp.n + min(sim_next, sp.n - 1)));  // seq-halving target -> s_misc[0]
    // backward operands of levels hl and hl + 16: visits, value, variance -> s_back[32 / 64 / 96 + lev]
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int lev = hl + kStaged2Lanes * k;
      if (lev >= L) break;
      const uint32_t* nrec = reinterpret_cast<const uint32_t*>(t.nodes + ((s_back[lev] & 0xffffu) * uB + ub));
      const uint32_t d = smem_u32(s_back + 32 + lev);
      cp_async4(d, nrec + 0);
      cp_async4(d + 4u * 32, nrec + 1);
      cp_async4(d + 4u * 64, nrec + 2);
    }
    // words 0..8 of staged2_store_lane's record of (path level r * kPR + glev, action gl) in round r
    if (gl < t.A) {
#pragma unroll
      for (int r = 0; r < kRounds; ++r) {
        const int lev = r * kPR + glev;
        if (lev >= L) break;
        const unsigned slot_g = (s_back[lev] & 0xffffu) * uB + ub;
        const uint32_t* erec = reinterpret_cast<const uint32_t*>(t.edges + (size_t)(slot_g * uA + (unsigned)gl));
        const uint32_t* nrec = reinterpret_cast<const uint32_t*>(t.nodes + slot_g);
        const uint32_t d = smem_u32(s_edge + r * kStaged2LaneWords * kStaged2Lanes + hl);
#pragma unroll
        for (int k = 0; k < 7; ++k) cp_async4(d + 4u * kStaged2Lanes * k, erec + k);  // ci1, vis, pl, rew, val, vvar, dis
        cp_async4(d + 4u * kStaged2Lanes * 7, nrec + 4);                            // raw value, raw variance (node half 1)
        cp_async4(d + 4u * kStaged2Lanes * 8, nrec + 5);
      }
    }
  };
  // ---- stage the records the step for simulation `sim_next` will need (tree_step2_kernel's pre-wait staging).  issued: the copies
  // are in flight (after a descent); otherwise the path comes from a DIRECT step and resync, and they are issued here.
  auto stage = [&](int sim_next, bool issued) {
    if (!issued) issue_staging(sim_next);
    staged = __all_sync(0xffffffffu, !in_batch || stageable(sim_next));
    cp_async_wait_all();
    __syncwarp();
    if (!staged) return;
    const int Lw = max(L, __shfl_xor_sync(0xffffffffu, L, kStaged2Lanes));
#pragma unroll
    for (int r = 0; r < kRounds; ++r) {
      if (r * kPR <= Lw) {  // warp-uniform
        const int lev = r * kPR + glev;
        const bool on = in_batch && lev <= L && gl < t.A;
        uint32_t* const se = s_edge + r * kStaged2LaneWords * kStaged2Lanes + hl;
        const float xl[1] = {on && lev < L ? __uint_as_float(se[2 * kStaged2Lanes]) : 0.0f};
        float pr[1];
        group_softmax<kG, 1>(xl, valid1, pr);  // p = max(tiny, softmax(prior logits)) of _compute_mixed_value
        if (on) {
          if (lev == L) {  // the fresh leaf's records are all zero
#pragma unroll
            for (int k = 0; k < 9; ++k) se[kStaged2Lanes * k] = 0u;
          }
          se[kStaged2Lanes * 9] = __float_as_uint(eaz_max(EAZ_F32_TINY, pr[0]));
        }
      }
    }
    __syncwarp();
  };

  // ---- simulation 0: the root's first selection + descent (DIRECT), then mirror the result
  direct_pair(a, 0, 0, 1, b0, lane);
  resync(0);
  {  // the root's score terms never change (mctx seq_halving.score_considered); lanes hl = 0 .. A-1 of the tree form its group 0
    const bool rt = in_batch && hl < t.A;
    const float lg = rt ? t.edges[(size_t)(ub * uA + (unsigned)hl)].pl : -INFINITY;  // root prior logits (max-subtracted / masked by root_init)
    const bool inval = rt && a.invalid && a.invalid[ub * uA + hl] != 0;
    const float m = group_max<kG>(lg);
    const int nvalid = group_sum_i<kG>((rt && !inval) ? 1 : 0);
    if (rt) {
      s_root[hl] = __float_as_uint(__fadd_rn(t.gumbel[ub * uA + hl], __fsub_rn(lg, m)));
      s_root[2 + hl] = inval ? 1u : 0u;
      if (hl == 0) s_misc[1] = (uint32_t)min(sp.max_considered, nvalid);
    }
  }
  __syncwarp();
  stage(1, false);

#pragma unroll 1
  for (int it = 0; it < n; ++it) {
    const int sim = it + 1;
    const bool do_select = sim < n;
    // lane a of a tree holds action a's logit (A <= kG = 2)
    const float lg = (in_batch && hl < t.A) ? (hl == 0 ? net.z : net.w) : -INFINITY;
    if (!staged) {  // DIRECT for both trees (reads the network outputs and the pending descent from the workspace)
      if (in_batch) {
        if (hl < t.A) t.net_logits[ub * uA + hl] = lg;
        if (hl == 0) {
          t.net_value[b] = net.x;
          t.net_ube[b] = net.y;
        }
      }
      __syncwarp();
      if (trc.buf && lane == 0) trc.path(it, tw, 0, 1);
      direct_pair(a, sim, 1, do_select ? 1 : 0, b0, lane);
      if (do_select) {
        resync(sim);
        stage(sim + 1, false);
      }
      continue;
    }

    // ---- 1. expand, 2. backward, 3. refresh (tree_step.cuh)
    const Staged2Leaf f = staged2_expand<kG>(t, sp, w, L, leaf, reward, lg, in_batch ? net.x : 0.0f, in_batch ? net.y : 0.0f, term);
    if (lane == 0) trc.stamp(it, tw, 0);
    staged2_backward<kG>(t, w, f, std_backup);
    if (lane == 0) trc.stamp(it, tw, 1);
    if (!do_select) continue;  // the last step only completes the backward
    staged2_refresh<kG>(t, sp, w, f, beta, s_root, s_root + 2, s_misc, s_next);
    if (lane == 0) trc.stamp(it, tw, 2);

    // ---- 4. simulate: follow the cached selections (all 16 lanes of a tree run the same chase), then the DeepSea transition
    {
      // (32-bit shared addresses taken through a shuffle + loop-invariant operands in registers: written with the generic pointers,
      // every level re-derived the shared window base -- S2UR SR_CgaCtaId -- and re-read B / max_depth / the path pointer from the
      // constant bank, ~290 cycles per level on the critical path; C2 0.961 -> 0.947 ms / step)
      int node = 0, depth = 0, action = 0, child = -1;
      bool active = in_batch;
      const int max_depth = sp.max_depth;
      int2* path_p = t.path + ub;
      const uint32_t next_sa = opaque_u32(smem_u32(s_next));
      uint32_t back_p = opaque_u32(smem_u32(s_back));
      while (__any_sync(0xffffffffu, active)) {
        if (active) {
          const int nx = (int)lds_u16(next_sa + 2u * (uint32_t)node);
          action = nx & 3;
          child = (nx >> 2) - 1;
          if (hl == 0) {
            *path_p = make_int2(node, action);
            if (depth < 32) sts_u32(back_p, (uint32_t)node | ((uint32_t)action << 16));
          }
          path_p += uB;
          back_p += 4u;
          depth += 1;
          if (child < 0 || depth >= max_depth) active = false;
          else node = child;
        }
      }
      __syncwarp();  // (lane 0's s_back words of the path -> the lanes that issue the staging copies)
      if (in_batch) {
        L = depth;
        leaf = child < 0 ? sim + 1 : child;  // search.py: node first expanded on simulation i gets index i+1
      }
      issue_staging(sim + 1);
      if (in_batch) {
        float rw;
        const uint32_t ns = deepsea_step(s_state[node], action, a.env.size, amap_n ? s_amap : a.env.action_map, &rw);  // context.py:127 env.step fused here
        net = __ldg(a.ds_out + deepsea_obs_index(ns, a.env.size));  // the new leaf's network outputs: in flight with the staging copies
        reward = rw;
        term = EAZ_DS_TERM(ns) != 0;
        if (hl == 0) {
          t.path_len[b] = depth;
          t.parent[b] = node;
          t.action[b] = action;
          t.leaf[b] = leaf;
          t.reward[b] = rw;
          st_global[(unsigned)leaf * uB + ub] = ns;
          if (leaf < ncap) s_state[leaf] = ns;
        }
      }
      __syncwarp();
    }
    if (trc.buf) {
      const int Lmax = max(L, __shfl_xor_sync(0xffffffffu, L, kStaged2Lanes));
      if (lane == 0) {
        trc.stamp(it, tw, 3);
        trc.path(it, tw, Lmax, 0);
      }
    }
    stage(sim + 1, true);
    if (lane == 0) trc.stamp(it, tw, 4);
  }
}

}  // namespace ps
}  // namespace eaz
