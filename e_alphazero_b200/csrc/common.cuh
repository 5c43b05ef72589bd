// common.cuh -- shared device code of libeaz_b200: error plumbing, the compact
// in-tree env-state encodings, the DeepSea / Subleq transitions, the XXHash
// variant, and the lane-group reductions whose order is the contract with the
// CPU oracle (oracle/eaz_oracle.c: orc_tree_sum).
#pragma once
#include <cstdlib>

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/eaz_b200.h"
#include "../../include/eaz_math.h"

namespace eaz {

// ---------------------------------------------------------------- errors
void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define EAZ_CHECK_ARG(cond, ...)      \
  do {                                \
    if (!(cond)) {                    \
      ::eaz::set_error(__VA_ARGS__);  \
      return EAZ_ERR_INVALID_ARG;     \
    }                                 \
  } while (0)

#define EAZ_CHECK_LAUNCH(what)                                   \
  do {                                                           \
    cudaError_t e__ = cudaGetLastError();                        \
    if (e__ != cudaSuccess) return ::eaz::cuda_fail(e__, what);  \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Optional launch timeline (eaz_debug_set_timeline): block 0 of the per-simulation kernels appends
// {globaltimer at entry, after the PDL wait, at exit, kind} records; tl[0] is the record counter.
extern unsigned long long* g_timeline;
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// Programmatic dependent launch (PDL): the kernel may start while its predecessor in the stream is still running;
// everything before pdl_wait() must not touch data the predecessor produces.  pdl_trigger() lets the successor start.
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// Per-tile completion counters (search.cu "tile flags"): a finer-grained replacement for the grid-wide PDL wait between the
// tree kernel and the network kernel of the fused DeepSea path.  Producers make their results visible (fence) and bump the
// counter of their 128-tree tile; consumers poll it with acquire loads.  Counters only grow within a search (zeroed at its
// start), so a launch waits for `>= epoch * producers_per_tile`.  The spin is bounded: a protocol bug traps instead of hanging.
constexpr int kTileRows = 128;
__device__ __forceinline__ int ld_relaxed_gpu(const int* p) {
  int v;
  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// ONE thread polls (relaxed loads straight from L2, with a back-off) and then issues the acquire fence; the caller
// releases the rest of the CTA / warp with a barrier.  Hundreds of pollers or an acquire per poll would flood the memory pipe.
__device__ __forceinline__ void wait_counter(const int* ctr, int target) {
  unsigned spins = 0;
  while (ld_relaxed_gpu(ctr) < target) {
    __nanosleep(100);
    if (++spins > (1u << 24)) __trap();
  }
  __threadfence();
}
__device__ __forceinline__ void signal_counter(int* ctr) {  // caller: results written, __syncwarp / __syncthreads done
  asm volatile("fence.acq_rel.gpu;" ::: "memory");
  asm volatile("red.relaxed.gpu.global.add.s32 [%0], 1;" ::"l"(ctr) : "memory");
}

template <typename... KArgs, typename... Args>
static inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  static const int no_pdl = getenv("EAZ_NO_PDL") != nullptr;  // measurement / debugging knob: plain stream order (no early launch)
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = no_pdl ? 0 : 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}

// Internal eaz_search_config.flags bit (set by eaz_evaluate / eaz_selfplay, never by a caller): enqueue only the search's preparation -- the tree
// memset, the root states and, unless EAZ_FLAG_REUSE_PREPARED, the parameter-derived tables -- and no simulation.
constexpr int kFlagPrepareOnly = 1 << 28;

// ---------------------------------------------------------------- env description (by value into kernels)
struct EnvDesc {
  int kind;
  int size;                   // DeepSea N
  const uint8_t* action_map;  // device, may be null
  int ws;                     // Subleq word size
  int binary;
  int reward_fn;
  int obs_cols;   // N | bit width | ws+1
  int obs_dim;    // flattened observation length
  int num_actions;
  int compact_bytes;
};

inline int binary_width(int ws) {  // envs/subleq.py:59-60
  int x = ws - 1, n = 0;
  while (x > 0) { n++; x >>= 1; }
  return n + 1;
}

int make_env_desc(const eaz_env* env, EnvDesc* d);  // validates like the reference asserts

// Pointers of an eaz_state, by value.
struct StateSoA {
  int32_t* step_count;
  float* rewards;
  uint8_t* terminated;
  uint8_t* truncated;
  uint8_t* observation;
  int32_t* col;
  int32_t* memory;
  int32_t* task;
  uint8_t* solved;
  int32_t* input_after;
  int32_t* output_after;
};
inline StateSoA soa_of(const eaz_state* s) {
  return StateSoA{s->step_count, s->rewards, s->terminated, s->truncated, s->observation, s->col,
                  s->memory, s->task, s->solved, s->input_after, s->output_after};
}

// ---------------------------------------------------------------- compact states
// DeepSea: one u32 -- bits 0..11 _step_count, 12..23 _horizontal_position,
// 24 terminated, 25 truncated.
// Subleq: [u16 in_after[8]] [u16 out_after[8]] [u16 step_count] [u8 task]
// [u8 flags: 1 terminated, 2 truncated, 4 solved] [4 reserved] [u8 memory[ws]]
// padded to a multiple of 8 bytes (40 + roundup8(ws)).
#define EAZ_DS_STEP(v) ((int)((v)&0xfffu))
#define EAZ_DS_COL(v) ((int)(((v) >> 12) & 0xfffu))
#define EAZ_DS_TERM(v) ((int)(((v) >> 24) & 1u))
#define EAZ_DS_TRUNC(v) ((int)(((v) >> 25) & 1u))
__host__ __device__ inline uint32_t ds_pack(int step, int col, int term, int trunc) {
  return ((uint32_t)step & 0xfffu) | (((uint32_t)col & 0xfffu) << 12) | ((uint32_t)(term != 0) << 24) |
         ((uint32_t)(trunc != 0) << 25);
}

#define EAZ_SQ_HDR 40
#define EAZ_SQ_FLAG_TERM 1
#define EAZ_SQ_FLAG_TRUNC 2
#define EAZ_SQ_FLAG_SOLVED 4

// pgx.State leaves of env b -> its compact record at `out` (eaz_env_compact; the replay ring's add writes the same records)
__device__ __forceinline__ void pack_state(const EnvDesc& env, const StateSoA& s, int b, uint8_t* out) {
  const int term = s.terminated[b] != 0, trunc = s.truncated ? (s.truncated[b] != 0) : 0;
  if (env.kind == EAZ_ENV_DEEPSEA) {
    reinterpret_cast<uint32_t*>(out)[b] = ds_pack(s.step_count[b], s.col[b], term, trunc);
    return;
  }
  const int S = env.compact_bytes, ws = env.ws;
  uint8_t* o = out + (size_t)b * S;
  uint16_t* h = reinterpret_cast<uint16_t*>(o);
  for (int i = 0; i < 8; ++i) {
    h[i] = (uint16_t)s.input_after[(size_t)b * 8 + i];
    h[8 + i] = (uint16_t)s.output_after[(size_t)b * 8 + i];
  }
  h[16] = (uint16_t)s.step_count[b];
  o[34] = (uint8_t)s.task[b];
  o[35] = (uint8_t)((term ? EAZ_SQ_FLAG_TERM : 0) | (trunc ? EAZ_SQ_FLAG_TRUNC : 0) | (s.solved[b] ? EAZ_SQ_FLAG_SOLVED : 0));
  o[36] = o[37] = o[38] = o[39] = 0;
  for (int i = 0; i < S - EAZ_SQ_HDR; ++i) o[EAZ_SQ_HDR + i] = i < ws ? (uint8_t)s.memory[(size_t)b * ws + i] : 0;
}

// One 16-byte trajectory record of env b for the replay buffer's wire format (SURVEY 8f-3, main.py:383-385; eaz_trajectory_pack and
// the stacked outputs of eaz_selfplay): the played action, the reward bits, terminated | truncated << 8 | solved << 16, and the first
// word of the compact state (DeepSea: the whole state; Subleq: step count | task << 16 -- the memory image travels separately when the
// caller stores full states).
__device__ __forceinline__ int4 pack_trajectory(const EnvDesc& env, const StateSoA& s, const int32_t* __restrict__ action, int b) {
  const int term = s.terminated[b] != 0, trunc = s.truncated ? (s.truncated[b] != 0) : 0;
  int flags = term | (trunc << 8), word;
  if (env.kind == EAZ_ENV_DEEPSEA) {
    word = (int)ds_pack(s.step_count[b], s.col[b], term, trunc);
  } else {
    flags |= (s.solved[b] != 0) << 16;
    word = (s.step_count[b] & 0xffff) | (s.task[b] << 16);
  }
  return make_int4(action[b], __float_as_int(s.rewards[b]), flags, word);
}

// pgx.Env.step around DeepSea._step (deep_sea.py:59-81).  Returns the new
// packed state; *reward receives rewards[0].
__device__ __forceinline__ uint32_t deepsea_step(uint32_t s, int action, int N, const uint8_t* __restrict__ amap,
                                                 float* reward) {
  if (EAZ_DS_TERM(s) | EAZ_DS_TRUNC(s)) {  // absorbing: same state, zero rewards (pgx core.py Env.step)
    *reward = 0.0f;
    return s;
  }
  const int step = EAZ_DS_STEP(s) + 1;  // _step_count incremented before _step
  int col = EAZ_DS_COL(s);
  int row = min(max(step - 1, 0), N - 1);
  const int flip = amap ? (amap[row * N + min(col, N - 1)] != 0) : 0;  // :62
  const int shift = ((action == 0) != (flip != 0)) ? -1 : 1;          // :63
  col = min(max(col + shift, 0), N - 1);                               // :64
  const int term = step >= N - 1;                                      // :72
  *reward = (term && col == N - 1) ? 1.0f : 0.0f;                      // :74-78
  return ds_pack(step, col, term, 0);
}

// Observation cell of a DeepSea state (deep_sea.py:56,68-70).
__device__ __forceinline__ int deepsea_obs_index(uint32_t s, int N) {
  return min(EAZ_DS_STEP(s), N - 1) * N + EAZ_DS_COL(s);
}

// ---------------------------------------------------------------- Subleq test cases (subleq.py:398-501)
struct SubleqVec {
  int8_t len;
  int8_t v[8];
};
// [task 0..5][test 0..2]; the sixth row is the last lax.switch branch (MULTIPLICATION).
#define EAZ_SQ_IN_TABLE { \
    {{7, {1, 2, 3, 4, 5, 6, 7, 0}}, {8, {5, 4, 4, 5, 1, 2, 3, 1}}, {8, {1, 1, 6, 2, 4, 4, 5, 3}}}, \
    {{8, {-4, -3, -2, -1, 0, 1, 2, 3}}, {7, {1, 2, 3, 4, 5, 6, 7, 0}}, {5, {0, -1, 2, -3, 4, 0, 0, 0}}}, \
    {{8, {-4, -3, -2, -1, 0, 1, 2, 3}}, {7, {1, 2, 3, 4, 5, 6, 7, 0}}, {5, {0, -1, 2, -3, 4, 0, 0, 0}}}, \
    {{6, {1, 1, 5, 4, 0, -3, 0, 0}}, {6, {2, 3, 0, 0, -1, -2, 0, 0}}, {8, {1, 2, 3, 4, 4, 3, 2, 1}}}, \
    {{6, {1, 1, 5, 4, 0, -3, 0, 0}}, {6, {2, 3, 0, 0, -1, -2, 0, 0}}, {8, {1, 2, 3, 4, 4, 3, 2, 1}}}, \
    {{6, {1, 2, 2, 3, -7, 4, 0, 0}}, {6, {-1, -5, 5, 2, 0, 1, 0, 0}}, {6, {0, 0, 1, 1, -3, 3, 0, 0}}}, \
}
#define EAZ_SQ_OUT_TABLE { \
    {{7, {-1, -2, -3, -4, -5, -6, -7, 0}}, {8, {-5, -4, -4, -5, -1, -2, -3, -1}}, {8, {-1, -1, -6, -2, -4, -4, -5, -3}}}, \
    {{8, {4, 3, 2, 1, 0, -1, -2, -3}}, {7, {-1, -2, -3, -4, -5, -6, -7, 0}}, {5, {0, 1, -2, 3, -4, 0, 0, 0}}}, \
    {{8, {-4, -3, -2, -1, 0, 1, 2, 3}}, {7, {1, 2, 3, 4, 5, 6, 7, 0}}, {5, {0, -1, 2, -3, 4, 0, 0, 0}}}, \
    {{3, {0, 1, 3, 0, 0, 0, 0, 0}}, {3, {-1, 0, 1, 0, 0, 0, 0, 0}}, {4, {-1, -1, 1, 1, 0, 0, 0, 0}}}, \
    {{3, {2, 9, -3, 0, 0, 0, 0, 0}}, {3, {5, 0, -3, 0, 0, 0, 0, 0}}, {4, {3, 7, 7, 3, 0, 0, 0, 0}}}, \
    {{3, {2, 6, -28, 0, 0, 0, 0, 0}}, {3, {5, 10, 0, 0, 0, 0, 0, 0}}, {3, {0, 1, -9, 0, 0, 0, 0, 0}}}, \
}
static __constant__ SubleqVec c_sq_in[6][3] = EAZ_SQ_IN_TABLE;
static __constant__ SubleqVec c_sq_out[6][3] = EAZ_SQ_OUT_TABLE;
// The same vectors for word size 16, reduced mod 16 and packed one byte per element (sq_pack_vec's format) at COMPILE time:
// subleq_simulate16 reads two 64-bit constants instead of packing 16 elements (a modulo each) per call.
struct SqPacked16 {
  unsigned long long in[6][3], out[6][3];
};
constexpr unsigned long long sq_pack16_ce(const SubleqVec& v) {
  unsigned long long p = 0ull;
  for (int i = 0; i < 8; ++i)
    if (i < v.len) p |= (unsigned long long)(unsigned)(((int)v.v[i] % 16 + 16) % 16) << (8 * i);
  return p;
}
constexpr SqPacked16 sq_make_packed16() {
  constexpr SubleqVec tin[6][3] = EAZ_SQ_IN_TABLE;
  constexpr SubleqVec tout[6][3] = EAZ_SQ_OUT_TABLE;
  SqPacked16 p{};
  for (int r = 0; r < 6; ++r)
    for (int k = 0; k < 3; ++k) {
      p.in[r][k] = sq_pack16_ce(tin[r][k]);
      p.out[r][k] = sq_pack16_ce(tout[r][k]);
    }
  return p;
}
static __constant__ SqPacked16 c_sq16 = sq_make_packed16();

__host__ __device__ inline int floormod(int x, int m) {
  int r = x % m;
  return r < 0 ? r + m : r;
}
__device__ __forceinline__ int sq_task_row(int task) { return min(max(task - 1, 0), 5); }  // lax.switch clamps
// element i of test k: x % ws, padded with ws (subleq.py:402-404)
__device__ __forceinline__ int sq_test_in(int trow, int k, int i, int ws) {
  return i < c_sq_in[trow][k].len ? floormod(c_sq_in[trow][k].v[i], ws) : ws;
}
__device__ __forceinline__ int sq_test_out(int trow, int k, int i, int ws) {
  return i < c_sq_out[trow][k].len ? floormod(c_sq_out[trow][k].v[i], ws) : ws;
}

// One simulate() call (subleq.py:156-395) on a byte memory image living in
// shared or local memory.  `mem` is modified.  Returns correct / fills results.
struct SubleqSim {
  int in[8];
  int out[8];
  int bytes_used;
  int cycles;
  int correct;
};
// Words are < 256, so a test vector (8 words) is one 64-bit register: byte i = element i.
__device__ __forceinline__ unsigned long long sq_pack_vec(const SubleqVec& v, int ws) {
  unsigned long long p = 0ull;
#pragma unroll
  for (int i = 0; i < 8; ++i)
    if (i < v.len) p |= (unsigned long long)(unsigned)floormod(v.v[i], ws) << (8 * i);
  return p;
}
// The interpreter keeps the input as (packed vector, cursor), the output as (packed bytes, count), and the "output == expected"
// test as `no mismatch so far && count == expected length` (a written word is < ws, so it can never equal the pad token ws: the
// arrays are equal iff exactly the expected words were written and all matched).  Results are expanded into SubleqSim at the end.
// The loop body is branch-free apart from its exits (selects and predicated stores): the 32 lanes of a warp interpret 32 different
// programs.  Loads go to clamped (always valid) addresses and are discarded by selects.
//
// CYCLE DETECTION (exact).  43 % of the programs a search visits never halt and never err: the reference lets them spin until
// MAX_CYCLE_COUNT = 200 (subleq.py:19,297-299).  Everything that determines the machine's future -- memory, program counter, input
// cursor, output count (`bad` is 0 while running: a mismatch errs at once) -- is a deterministic function of itself, so when that
// state recurs the machine is in a loop it can never leave: it runs to the cap without halting or erring, its outputs / consumed
// inputs (monotone counters that were equal at both ends of the loop) and bytes_used (a running max that has already seen every
// instruction of the loop) are final, and `correct` is false (a program that has produced the expected output halts, :340-345).
// So the result equals the reference's with cycles = 200, and the remaining iterations are skipped.  Recurrence is found with
// Brent's algorithm against ONE snapshot (taken at cycles 0, 1, 2, 4, 8, ...): `diff` counts the bytes in which memory differs from
// the snapshot and is updated incrementally by the single store of each cycle, so the check costs one extra load per cycle for any
// word size.  Measured on the states of a C3 search: mean executed cycles 88 -> 5.3, worst lane of a warp 194 -> 22.
// `snap`: ws bytes of scratch next to `mem` (kDetect = false: the plain loop, `snap` unused).
// shared-memory byte accesses as opaque 32-bit operations: the compiler neither narrows the interpreter's arithmetic to 16-bit
// registers (PRMT / LOP3 packing on the dependence chain) nor reorders them -- their order below IS the issue order
__device__ __forceinline__ uint32_t sq_lds8(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}
__device__ __forceinline__ void sq_sts8(uint32_t addr, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(addr), "r"(v) : "memory"); }

// `mem`, `snap`: shared memory, sq_img_stride(ws) bytes each (>= ws + 4: a fetch at any reachable program counter stays inside).
template <bool kDetect>
__device__ __forceinline__ void subleq_simulate(int ws, uint8_t* mem, uint8_t* snap, int trow, int k, SubleqSim& r) {
  const int AMAX = ws - 4, AIN = ws - 3, AOUT = ws - 2;
  const unsigned half1 = (unsigned)((ws + 1) >> 1) - 1u;  // jump <=> value == 0 || 2 * value >= ws <=> (unsigned)(value - 1) >= ceil(ws / 2) - 1
  const int in_len = c_sq_in[trow][k].len, out_len = c_sq_out[trow][k].len;
  const unsigned long long tin = sq_pack_vec(c_sq_in[trow][k], ws), tout = sq_pack_vec(c_sq_out[trow][k], ws);
  const uint32_t m0 = (uint32_t)__cvta_generic_to_shared(mem), s0 = (uint32_t)__cvta_generic_to_shared(snap);
  unsigned long long outp = 0ull;
  int in_cur = 0, out_cur = 0, cur = 0, bytes = 0, cycles = 0, err = 0, bad = 0;
  // Brent: the snapshot is the state after 0, 1, 2, 4, 8, ... cycles (initially the start state: the caller passes snap == copy of mem)
  int diff = 0, lam = 0, pw = 1;
  uint32_t io_meta = 0u, snap_meta = 0u;  // io_meta = in_cur << 16 | out_cur << 20; a state's meta word = cur | io_meta
  bool hit = false;
  const int nwords = (ws + 3) >> 2;
  // One cycle's dependence chain is fetch (a, b, c) -> load operands -> subtract / wrap -> store, jump test -> next fetch: two
  // shared-memory round trips (29 cycles each) and ~8 ALU operations.  The few programs that really run to the cap set the kernel's
  // duration, and their warp runs alone on its scheduler, so the loop is built for LATENCY:
  //   * the operand loads go out (to clamped, always valid addresses) before anything is decided about the cycle, and the next
  //     fetch goes out as soon as the program counter is known -- both branches of the loop resolve under a load's latency;
  //   * the COMMON cycle (both operands plain memory cells, program counter in range, no snapshot due: nothing but the
  //     subtraction can happen, :322-329) takes a short path without any IO / error / halt bookkeeping;
  //   * the loop detector hangs off the chain (one extra load, a few compares).
  // (Measured per cycle, one warp alone: 120 ns for the first transcription, 190 ns with early-out branches on the chain or with a
  // generic-pointer null test in the loop -- S2UR every iteration --, see profiles/r2_summary.md for this version.)
  bool oob = false;  // cur + 2 >= ws (:364-370: costs a cycle, sets the error, changes nothing else); never at cur = 0 (ws >= 16)
  uint32_t a = sq_lds8(m0), b = sq_lds8(m0 + 1), c = sq_lds8(m0 + 2);
  while (true) {  // :297-299
    // ---- the tight loop: consecutive COMMON cycles, ~40 instructions each.  The operand loads go out (to clamped, always valid
    // addresses) BEFORE the cycle is classified, so the exit test resolves under their latency and the chain is
    // fetch -> clamp -> operand loads -> subtract, wrap -> jump test -> fetch; the back edge is unconditional.
    uint32_t am, bm;
    int ma, mb, sv;
    while (true) {
      am = min(a, (uint32_t)AMAX);
      bm = min(b, (uint32_t)AMAX);
      ma = (int)sq_lds8(m0 + am);
      mb = (int)sq_lds8(m0 + bm);
      sv = kDetect ? (int)sq_lds8(s0 + am) : 0;
      if (!(max(a, b) <= (uint32_t)AMAX && !oob && (!kDetect || lam + 1 != pw) && !hit && cycles < EAZ_SUBLEQ_MAX_CYCLES)) break;
      cycles += 1;
      const int dlt = ma - mb;  // both in [0, ws): floor-mod is one conditional add
      const int value = (int)min((unsigned)dlt, (unsigned)(dlt + ws));
      sq_sts8(m0 + am, (uint32_t)value);
      const int cur_n = ((unsigned)(value - 1) >= half1) ? (int)min(c, (uint32_t)(ws - 1)) : cur + 3;  // :329
      const uint32_t fa = m0 + (uint32_t)cur_n;  // cur_n <= ws: the fetch stays inside the image even when the next cycle is out of range
      a = sq_lds8(fa);
      b = sq_lds8(fa + 1);
      c = sq_lds8(fa + 2);
      bytes = max(bytes, cur + 3);  // :311
      cur = cur_n;
      oob = cur_n + 2 >= ws;
      if (kDetect) {
        diff += (int)(value != sv) - (int)(ma != sv);
        lam += 1;
        hit = diff == 0 && ((uint32_t)cur_n | io_meta) == snap_meta;  // the state after this cycle == the snapshot
      }
    }
    if (hit || cycles >= EAZ_SUBLEQ_MAX_CYCLES) break;
    // ---- the general cycle: an operand is IN / OUT / HALT, the program counter ran out of range, or a snapshot is due
    // (operands already loaded above, from the clamped addresses)
    cycles += 1;
    const bool live = !oob;
    const bool have_in = in_cur < in_len;  // input_state[0] < word_size (:197,218)
    const int in0 = have_in ? (int)((unsigned)(tin >> (8 * in_cur)) & 0xffu) : 0;
    const bool a_mem = a <= (uint32_t)AMAX, b_mem = b <= (uint32_t)AMAX, a_in = a == (uint32_t)AIN, b_in = b == (uint32_t)AIN;
    const int va = a_mem ? ma : (a_in ? in0 : 0);  // reads of OUT / HALT give 0 (:225-228)
    const int vb = b_mem ? mb : (b_in ? in0 : 0);
    const int dlt = va - vb;
    const int value = (int)min((unsigned)dlt, (unsigned)(dlt + ws));
    const bool wr = live && a_mem;  // writes to IN / HALT are ignored (:277-278,290-291)
    if (wr) {
      sq_sts8(m0 + am, (uint32_t)value);
      diff += (int)(value != sv) - (int)(ma != sv);
    }
    const int cur_n = live ? (((unsigned)(value - 1) >= half1) ? (int)min(c, (uint32_t)(ws - 1)) : cur + 3) : cur;
    const bool uses_in = a_in || b_in;
    const bool to_out = live && a == (uint32_t)AOUT;
    const bool out_ok = to_out && out_cur < 8;  // a write to a full output is an error (:282-283)
    const bool last_ok = !out_ok || (out_cur < out_len && value == (int)((unsigned)(tout >> (8 * out_cur)) & 0xffu));
    if (out_ok) {
      outp |= (unsigned long long)(unsigned)value << (8 * out_cur);
      out_cur += 1;
    }
    bad |= (out_ok && !last_ok) ? 1 : 0;
    in_cur += (live && uses_in && have_in) ? 1 : 0;  // :333-338 (at most one word per instruction)
    io_meta = ((uint32_t)in_cur << 16) | ((uint32_t)out_cur << 20);
    // :340-345 as written, `jump & c > AMAX`, parses as (jump & c) > AMAX = (c & 1) > ws - 4: never true for ws >= 16 -- the only
    // halt is "the expected output has been produced"
    const bool halt = live && !bad && out_cur == out_len;
    err = (oob || (live && uses_in && !have_in) || (to_out && !out_ok) || (out_ok && !last_ok)) ? 1 : 0;  // :346-350
    bytes = live ? max(bytes, cur + 3) : bytes;  // :311
    if (err || halt) break;
    if (kDetect) {
      hit = diff == 0 && ((uint32_t)cur_n | io_meta) == snap_meta;  // (against the current snapshot, before it is replaced)
      if (hit) break;
      if (++lam == pw) {  // new snapshot (the same cycles in every lane: 1, 2, 4, 8, ...)
        for (int i = 0; i < nwords; ++i) reinterpret_cast<uint32_t*>(snap)[i] = reinterpret_cast<const uint32_t*>(mem)[i];
        snap_meta = (uint32_t)cur_n | io_meta;
        diff = 0;
        lam = 0;
        pw <<= 1;
      }
    }
    const uint32_t fa = m0 + (uint32_t)cur_n;
    a = sq_lds8(fa);
    b = sq_lds8(fa + 1);
    c = sq_lds8(fa + 2);
    cur = cur_n;
    oob = cur_n + 2 >= ws;
  }
  if (hit && !err) cycles = EAZ_SUBLEQ_MAX_CYCLES;  // the reference's result after MAX_CYCLE_COUNT cycles is the current one
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    r.in[i] = (in_cur + i < in_len) ? (int)((tin >> (8 * (in_cur + i))) & 0xffull) : ws;
    r.out[i] = i < out_cur ? (int)((outp >> (8 * i)) & 0xffull) : ws;
  }
  r.bytes_used = bytes;
  r.cycles = cycles;
  r.correct = (!err) && !bad && out_cur == out_len;  // :394
}

// ---- word size 16 (the BASELINE Subleq configs C3 / C5): the whole machine in registers.
// Memory is 16 words of 4 bits = ONE 64-bit register (nibble i = mem[i]); a fetch is a shift, a store is a mask-and-insert, and the
// loop detector's snapshot is a second register compared as a whole (M == S) -- no shared memory, no `diff` counter, and the snapshot
// itself is free, so the tight loop takes the snapshots too.  The dependence chain of a common cycle is ~14 integer operations
// (fetch shift -> clamp -> operand shift -> subtract -> insert) against two shared-memory round trips + ~10 operations above.  Same
// cycle semantics, statement for statement (subleq.py:156-395); any snapshot schedule is exact (see CYCLE DETECTION above).
__host__ __device__ __forceinline__ unsigned long long sq_pack_nibbles16(const uint32_t* w4) {  // 16 bytes (each < 16) -> 16 nibbles
  unsigned long long m = 0ull;
  for (int i = 0; i < 4; ++i) {
    const uint32_t w = w4[i];
    const uint32_t n = (w & 0xFu) | ((w >> 4) & 0xF0u) | ((w >> 8) & 0xF00u) | ((w >> 12) & 0xF000u);
    m |= (unsigned long long)n << (16 * i);
  }
  return m;
}
template <bool kDetect>
__device__ __forceinline__ void subleq_simulate16(unsigned long long M, int trow, int k, SubleqSim& r) {
  constexpr int ws = 16, AMAX = ws - 4, AIN = ws - 3, AOUT = ws - 2;
  constexpr unsigned half1 = (unsigned)((ws + 1) >> 1) - 1u;
  const int in_len = c_sq_in[trow][k].len, out_len = c_sq_out[trow][k].len;
  const unsigned long long tin = c_sq16.in[trow][k], tout = c_sq16.out[trow][k];  // == sq_pack_vec(c_sq_in / c_sq_out[trow][k], 16)
  unsigned long long outp = 0ull, S = M;  // S: Brent's snapshot (initially the start state)
  int in_cur = 0, out_cur = 0, cur = 0, bytes = 0, cycles = 0, err = 0, bad = 0;
  int lam = 0, pw = 1;
  uint32_t io_meta = 0u, snap_meta = 0u;
  bool hit = false, oob = false;
  uint32_t f = (uint32_t)M;  // the three words at the program counter: nibbles 0..2
  while (true) {
    uint32_t a4, b4, am4, bm4;  // operand addresses, already times 4 (= bit offsets into M)
    int ma, mb;
    while (true) {  // consecutive COMMON cycles (both operands plain memory cells)
      a4 = (f << 2) & 0x3Cu;
      b4 = (f >> 2) & 0x3Cu;
      am4 = min(a4, (uint32_t)(4 * AMAX));
      bm4 = min(b4, (uint32_t)(4 * AMAX));
      ma = (int)((uint32_t)(M >> am4) & 15u);
      mb = (int)((uint32_t)(M >> bm4) & 15u);
      if (!(max(a4, b4) <= (uint32_t)(4 * AMAX) && !oob && !hit && cycles < EAZ_SUBLEQ_MAX_CYCLES)) break;
      cycles += 1;
      const int c = (int)((f >> 8) & 15u);
      const int seq = cur + 3;  // <= 16 (a cycle only runs at cur <= 13)
      const int value = (ma - mb) & 15;  // floor-mod 16 of a difference of two words
      M = (M & ~(15ull << am4)) | ((unsigned long long)(unsigned)value << am4);
      // both candidate fetches go out as soon as the store has landed; the jump test (:329) picks one.  An out-of-range fetch
      // (program counter >= 14) is never used (oob), so the shift count is only kept in range.
      const uint32_t f_jump = (uint32_t)(M >> (4 * c)), f_seq = (uint32_t)(M >> (4 * min(seq, 15)));
      const bool jump = (unsigned)(value - 1) >= half1;
      f = jump ? f_jump : f_seq;
      const int cur_n = jump ? c : seq;
      bytes = max(bytes, seq);  // :311
      cur = cur_n;
      oob = cur_n + 2 >= ws;
      if (kDetect) {
        const uint32_t meta = (uint32_t)cur_n | io_meta;
        hit = M == S && meta == snap_meta;
        if (++lam == pw) {  // (a hit leaves the loop before the new snapshot matters)
          S = M;
          snap_meta = meta;
          lam = 0;
          pw <<= 1;
        }
      }
    }
    if (hit || cycles >= EAZ_SUBLEQ_MAX_CYCLES) break;
    // ---- the general cycle: an operand is IN / OUT / HALT, or the program counter ran out of range
    cycles += 1;
    const uint32_t a = a4 >> 2, b = b4 >> 2;
    const int c = (int)((f >> 8) & 15u);
    const bool live = !oob;
    const bool have_in = in_cur < in_len;
    const int in0 = have_in ? (int)((unsigned)(tin >> (8 * in_cur)) & 0xffu) : 0;
    const bool a_mem = a <= (uint32_t)AMAX, b_mem = b <= (uint32_t)AMAX, a_in = a == (uint32_t)AIN, b_in = b == (uint32_t)AIN;
    const int va = a_mem ? ma : (a_in ? in0 : 0);
    const int vb = b_mem ? mb : (b_in ? in0 : 0);
    const int value = (va - vb) & 15;
    if (live && a_mem) M = (M & ~(15ull << am4)) | ((unsigned long long)(unsigned)value << am4);
    const int cur_n = live ? (((unsigned)(value - 1) >= half1) ? c : cur + 3) : cur;
    const bool uses_in = a_in || b_in;
    const bool to_out = live && a == (uint32_t)AOUT;
    const bool out_ok = to_out && out_cur < 8;
    const bool last_ok = !out_ok || (out_cur < out_len && value == (int)((unsigned)(tout >> (8 * out_cur)) & 0xffu));
    if (out_ok) {
      outp |= (unsigned long long)(unsigned)value << (8 * out_cur);
      out_cur += 1;
    }
    bad |= (out_ok && !last_ok) ? 1 : 0;
    in_cur += (live && uses_in && have_in) ? 1 : 0;
    io_meta = ((uint32_t)in_cur << 16) | ((uint32_t)out_cur << 20);
    const bool halt = live && !bad && out_cur == out_len;
    err = (oob || (live && uses_in && !have_in) || (to_out && !out_ok) || (out_ok && !last_ok)) ? 1 : 0;
    bytes = live ? max(bytes, cur + 3) : bytes;
    if (err || halt) break;
    if (kDetect) {
      const uint32_t meta = (uint32_t)cur_n | io_meta;
      hit = M == S && meta == snap_meta;
      if (hit) break;
      if (++lam == pw) {
        S = M;
        snap_meta = meta;
        lam = 0;
        pw <<= 1;
      }
    }
    f = (uint32_t)(M >> (4 * min(cur_n, 15)));
    cur = cur_n;
    oob = cur_n + 2 >= ws;
  }
  if (hit && !err) cycles = EAZ_SUBLEQ_MAX_CYCLES;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    r.in[i] = (in_cur + i < in_len) ? (int)((tin >> (8 * (in_cur + i))) & 0xffull) : ws;
    r.out[i] = i < out_cur ? (int)((outp >> (8 * i)) & 0xffull) : ws;
  }
  r.bytes_used = bytes;
  r.cycles = cycles;
  r.correct = (!err) && !bad && out_cur == out_len;
}

__device__ __forceinline__ float subleq_reward(int reward_fn, int solved, int bytes_used) {
  if (reward_fn == EAZ_SUBLEQ_REWARD_LOWEST_BYTES) return __fdiv_rn((float)solved, (float)(1 + bytes_used));  // :540-542
  return (float)solved;                                                                                      // :535-537
}

// ---------------------------------------------------------------- XXHash variant (network/hashes.py:162-229)
#define EAZ_XX_P1 0x9E3779B1u
#define EAZ_XX_P2 0x85EBCA77u
#define EAZ_XX_P3 0xC2B2AE3Du
#define EAZ_XX_ONE 0x3F800000u  // bit pattern of 1.0f
__device__ __forceinline__ uint32_t rotl32(uint32_t x, int n) { return __funnelshift_l(x, x, n); }
__device__ __forceinline__ uint32_t xx_init(int lane) {
  return lane == 0 ? 1u + EAZ_XX_P1 + EAZ_XX_P2 : lane == 1 ? 1u + EAZ_XX_P2 : lane == 2 ? 1u : 1u - EAZ_XX_P1;  // :217-220
}
__device__ __forceinline__ uint32_t xx_round(uint32_t acc, uint32_t word) {
  return rotl32(acc + word * EAZ_XX_P2, 13) * EAZ_XX_P1;  // :176-181
}
__device__ __forceinline__ uint32_t xx_finish(uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, int L, int bits) {
  uint32_t h = rotl32(a0, 1) + rotl32(a1, 7) + rotl32(a2, 12) + rotl32(a3, 18);  // :187
  h += (uint32_t)L;                                                              // :226
  h ^= h >> 15; h *= EAZ_XX_P2; h ^= h >> 13; h *= EAZ_XX_P3; h ^= h >> 16;      // :190-197
  return bits >= 32 ? h : (h >> (32 - bits));                                    // :229
}

// ---------------------------------------------------------------- lane groups
// G lanes per tree, action a in lane a % G, slot a / G.  Sums: slots ascending
// from 0.0f per lane, then xor-butterfly with strides 1,2,..,G/2.
template <int G>
__device__ __forceinline__ float group_sum(float v) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) v = __fadd_rn(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}
template <int G>
__device__ __forceinline__ int group_sum_i(int v) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
  return v;
}
template <int G>
__device__ __forceinline__ int group_max_i(int v) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}
template <int G>
__device__ __forceinline__ float group_max(float v) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}
template <int G>
__device__ __forceinline__ float group_min(float v) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, s));
  return v;
}
// argmax with lowest index among maxima (jnp.argmax)
template <int G>
__device__ __forceinline__ int group_argmax(float v, int idx) {
#pragma unroll
  for (int s = 1; s < G; s <<= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, v, s);
    const int oi = __shfl_xor_sync(0xffffffffu, idx, s);
    if (ov > v || (ov == v && oi < idx)) { v = ov; idx = oi; }
  }
  return idx;
}

}  // namespace eaz

// ---------------------------------------------------------------- Subleq step, block-cooperative
// A block of 3*EAZ_SQ_EPB threads advances EAZ_SQ_EPB envs: thread (e,k) runs
// test case k of env e (run_tests, subleq.py:504-532, vmaps the 3 tests).
#define EAZ_SQ_EPB 32
#define EAZ_SQ_IMG 264  // >= 256 + slack, multiple of 8
namespace eaz {
struct SqShared {
  alignas(16) uint8_t base[EAZ_SQ_EPB][EAZ_SQ_IMG];  // program after writing the action
  int16_t in_after[EAZ_SQ_EPB][8];
  int16_t out_after[EAZ_SQ_EPB][8];
  int correct[EAZ_SQ_EPB][3];
  int bytes[EAZ_SQ_EPB][3];
  int run[EAZ_SQ_EPB];   // 1 = execute the program for this env
  int trow[EAZ_SQ_EPB];  // row of the test-case table
};
// Per-(env, test) scratch in DYNAMIC shared memory: the memory image the test runs on and the cycle detector's snapshot of it.
// The stride is a whole number of words, odd in words whenever ws is a multiple of 8 (same-offset accesses of a warp: no conflicts).
__host__ __device__ inline int sq_img_stride(int ws) { return ((ws + 3) & ~3) + 4; }
__host__ __device__ inline size_t sq_dyn_smem_bytes(int ws) { return (size_t)2 * 3 * EAZ_SQ_EPB * sq_img_stride(ws); }
// launch helper: dynamic shared memory above 48 KB (ws > ~200) needs the opt-in attribute, set once per kernel
template <typename K>
inline cudaError_t sq_prepare_launch(K kernel, int ws, size_t* dyn_out) {
  const size_t dyn = sq_dyn_smem_bytes(ws);
  *dyn_out = dyn;
  if (dyn + sizeof(SqShared) + 1024 <= 48 * 1024) return cudaSuccess;
  return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sq_dyn_smem_bytes(256));
}

// All 3*EPB threads call this after base/run/trow are filled and synced; `dyn` = the kernel's dynamic shared memory
// (sq_dyn_smem_bytes).  On return (after its trailing __syncthreads) in_after/out_after/correct/bytes hold the results.
__device__ __forceinline__ void sq_run_tests_block(SqShared& sh, uint8_t* dyn, int ws) {
  const int e = threadIdx.x / 3, k = threadIdx.x % 3;
  if (sh.run[e]) {
    const uint32_t* base = reinterpret_cast<const uint32_t*>(sh.base[e]);
    SubleqSim r;
    if (ws == 16) {  // register-resident machine (no per-test image)
      subleq_simulate16<true>(sq_pack_nibbles16(base), sh.trow[e], k, r);
    } else {
      const int stride = sq_img_stride(ws);
      uint8_t* img = dyn + (size_t)threadIdx.x * stride;
      uint8_t* snap = dyn + (size_t)(3 * EAZ_SQ_EPB + threadIdx.x) * stride;
      for (int i = 0; i < (ws + 3) >> 2; ++i) {
        const uint32_t w = base[i];
        reinterpret_cast<uint32_t*>(img)[i] = w;
        reinterpret_cast<uint32_t*>(snap)[i] = w;  // the detector's first snapshot: the start state
      }
      subleq_simulate<true>(ws, img, snap, sh.trow[e], k, r);
    }
    sh.correct[e][k] = r.correct;
    sh.bytes[e][k] = r.bytes_used;
    if (k == 0) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        sh.in_after[e][i] = (int16_t)r.in[i];
        sh.out_after[e][i] = (int16_t)r.out[i];
      }
    }
  }
  __syncthreads();
}

// ---------------------------------------------------------------- pgx.Env.step on struct-of-arrays states (env.cu, evaluate.cu)
// DeepSea, one env per thread; auto_reset applies selfplay.py:66-71 to an env that is already terminal.
__device__ __forceinline__ void deepsea_state_step(const EnvDesc& env, const StateSoA& s, const int32_t* __restrict__ action, int auto_reset, int b) {
  const int term = s.terminated[b] != 0, trunc = s.truncated ? (s.truncated[b] != 0) : 0;
  if (auto_reset && (term | trunc)) {  // selfplay.py:66-71
    s.step_count[b] = 0;
    s.col[b] = 0;
    s.rewards[b] = 0.0f;
    s.terminated[b] = 0;
    if (s.truncated) s.truncated[b] = 0;
    return;
  }
  float reward;
  const uint32_t n = deepsea_step(ds_pack(s.step_count[b], s.col[b], term, trunc), action[b], env.size, env.action_map, &reward);
  s.step_count[b] = EAZ_DS_STEP(n);
  s.col[b] = EAZ_DS_COL(n);
  s.terminated[b] = (uint8_t)EAZ_DS_TERM(n);
  s.rewards[b] = reward;
}

// Subleq, EAZ_SQ_EPB envs per block of 3*EAZ_SQ_EPB threads (all of them call this; `dyn` = sq_dyn_smem_bytes of dynamic shared
// memory).  mode: 0 = init (task from task_ids), 1 = step, 2 = step with auto_reset.  On return thread (e, 0) has written env e's leaves.
__device__ __forceinline__ void subleq_block_step(const EnvDesc& env, const StateSoA& s, const int32_t* __restrict__ action,
                                                  const int32_t* __restrict__ task_ids, int mode, int B, SqShared& sh, uint8_t* dyn,
                                                  int* kind /* [EAZ_SQ_EPB] shared: 0 absorbing, 1 terminate now, 2 execute, 3 init/reset */) {
  const int ws = env.ws;
  const int e = threadIdx.x / 3, k = threadIdx.x % 3;
  const int b = blockIdx.x * EAZ_SQ_EPB + e;
  if (k == 0) {
    int kd = -1, run = 0;
    if (b < B) {
      const int term = s.terminated[b] != 0, trunc = s.truncated ? (s.truncated[b] != 0) : 0;
      if (mode == 0 || (mode == 2 && (term | trunc))) {
        const int task = task_ids ? task_ids[b] : (mode == 0 ? 1 : s.task[b]);
        s.task[b] = task;
        sh.trow[e] = sq_task_row(task);
        for (int i = 0; i < ws; i += 1) sh.base[e][i] = 0;  // empty program, subleq.py:630
        kd = 3;
        run = 1;
      } else if (term | trunc) {
        kd = 0;
      } else {
        const int step = s.step_count[b] + 1;
        s.step_count[b] = step;
        if (step >= ws - 3 || s.solved[b]) {  // subleq.py:671-673
          kd = 1;
        } else {
          sh.trow[e] = sq_task_row(s.task[b]);
          const int32_t* m = s.memory + (size_t)b * ws;
          for (int i = 0; i < ws; ++i) sh.base[e][i] = (uint8_t)m[i];
          sh.base[e][step - 1] = (uint8_t)action[b];  // :654
          kd = 2;
          run = 1;
        }
      }
    }
    kind[e] = kd;
    sh.run[e] = run;
  }
  __syncthreads();
  sq_run_tests_block(sh, dyn, ws);
  if (k != 0 || b >= B) return;
  const int kd = kind[e];
  if (kd == 0) {
    s.rewards[b] = 0.0f;
  } else if (kd == 1) {
    s.terminated[b] = 1;
    s.rewards[b] = 0.0f;
  } else if (kd >= 2) {
    const int solved = sh.correct[e][0] & sh.correct[e][1] & sh.correct[e][2];
    const int bytes = max(sh.bytes[e][0], max(sh.bytes[e][1], sh.bytes[e][2]));
    s.rewards[b] = subleq_reward(env.reward_fn, solved, bytes);
    s.solved[b] = (uint8_t)solved;
    int32_t* m = s.memory + (size_t)b * ws;
    if (kd == 3) {
      for (int i = 0; i < ws; ++i) m[i] = 0;
      s.step_count[b] = 0;
      s.terminated[b] = 0;
      if (s.truncated) s.truncated[b] = 0;
    } else {
      m[s.step_count[b] - 1] = action[b];
    }
    for (int i = 0; i < 8; ++i) {
      s.input_after[(size_t)b * 8 + i] = sh.in_after[e][i];
      s.output_after[(size_t)b * 8 + i] = sh.out_after[e][i];
    }
  }
}
}  // namespace eaz
