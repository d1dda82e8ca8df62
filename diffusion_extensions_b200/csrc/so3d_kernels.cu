// so3d_kernels.cu -- sm_100a kernels + C ABI (include/so3d.h) for the SO(3) diffusion hot path.
//
// Execution model (B200: 148 SMs, 64 warps/SM, 227 KB smem/CTA, HBM3e ~6.5 TB/s measured):
//   * one rotation per thread, all 3x3 math in registers, every op of a call fused in one kernel;
//   * rotations are 36-byte AoS records, so a warp reading "its" rows directly would touch each
//     128-byte line 9 times.  Instead a CTA moves a whole tile (kTile rows, contiguous in memory)
//     between HBM and shared memory with coalesced 16-byte vector accesses and each thread reads its
//     row from shared memory at a stride of 9 (or 3) words -- odd, hence bank-conflict free;
//   * grids are persistent: min(#tiles, 148 * CTAs/SM) CTAs striding over the tiles;
//   * HBM-bound kernels use streaming loads/stores (ld.global.cs / st.global.cs): nothing is re-read;
//   * the series evaluator is bound by FP32 operand bandwidth / MUFU / issue at once (7 FP32 + 1 MUFU.EX2 +
//     1 uniform constant load per term, see so3d_math.cuh).
// No library calls, no tensor cores (nothing here is GEMM shaped).
#include <cuda_runtime.h>
#include <stdio.h>
#include <type_traits>
#include <stdlib.h>
#include <string.h>

#include "../../include/so3d.h"
#include "so3d_math.cuh"
#include "so3d_lanes.cuh"
#include "so3d_tma.cuh"
#include "so3d_cdf_smem.cuh"

using namespace so3d;

namespace {

constexpr int kTile = 256;  // rows per tile == threads per CTA

// Build-time tuning knobs of the fused steps.  A variant library is built with
//   python tests/tools/build_variant.py NAME -DSO3D_QS_MINCTAS=5 ...
// and selected at run time with SO3D_LIB_PATH=build/variants/libso3d_NAME.so (tests/tools/probe_engine.py compares them);
// the defaults are the measured winners (profiles/r01l..r01u_probe_engine.jsonl).  Run-time aids: SO3D_ENGINE=cta|warp
// overrides the per-op schedule, SO3D_CTAS_PER_SM caps the persistent grid.
#ifndef SO3D_QS_OUTSTAGES
#define SO3D_QS_OUTSTAGES 1  // forward noising: output stages (1: more resident CTAs)
#endif
#ifndef SO3D_QS_MINCTAS
#define SO3D_QS_MINCTAS 4    // forward noising: resident CTAs promised to ptxas (4 -> <= 64 registers, no spills)
#endif
#ifndef SO3D_WROW_SHFL
#define SO3D_WROW_SHFL 1
#endif
#ifndef SO3D_QSX_MINCTAS
#define SO3D_QSX_MINCTAS 4   // forward noising with the noise / score outputs compiled in
#endif
#ifndef SO3D_PSS_OUTSTAGES
#define SO3D_PSS_OUTSTAGES 2 // shared-t reverse step: output stages
#endif
#ifndef SO3D_PSS_MINCTAS
#define SO3D_PSS_MINCTAS 1   // shared-t reverse step: no register cap (63 registers schedule 3 % faster than 48)
#endif
#ifndef SO3D_PS_MINCTAS
#define SO3D_PS_MINCTAS 3    // per-row-t reverse step (with the prefetch hooks: 3 -> 70 registers 0.418 ms, 4 -> 63 registers 0.423, 5 -> 48 + spills 0.455; r03z)
#endif

thread_local char g_err[256] = "";

int fail(int code, const char* what) {
  snprintf(g_err, sizeof(g_err), "%s", what);
  return code;
}

int check_launch(const char* name) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    snprintf(g_err, sizeof(g_err), "%s: %s", name, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

// Per-device caches (a process may drive several GPUs: kernel attributes such as the dynamic shared-memory limit are
// per device, so "configured once" must mean once per device).
constexpr int kMaxDevices = 64;
inline int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) d = 0;
  return d;
}
int g_sm_count[kMaxDevices] = {0};
int sm_count() {
  const int dev = current_device();
  if (g_sm_count[dev] == 0) {
    int n = 0;
    g_sm_count[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148;
  }
  return g_sm_count[dev];
}

inline int grid_for(int64_t n, int ctas_per_sm) {
  const int64_t tiles = (n + kTile - 1) / kTile;
  const int64_t cap = (int64_t)sm_count() * ctas_per_sm;
  return (int)(tiles < cap ? tiles : cap);
}

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ------------------------------------------------------------------------------------------------
// The row engine: one persistent, TMA-pipelined kernel template shared by every op.
//
//   Op provides
//     static constexpr int kIn9, kIn3, kOut9, kOut3  -- how many n x 9 / n x 3 arrays it reads / writes
//     const float* in9[kIn9], in3[kIn3]; float* out9[kOut9], out3[kOut3]   (an output may be NULL = skipped)
//     static constexpr int kTab;  __device__ void setup(float* tab) const   -- CTA-shared tables (CDF row, guide, ...)
//     __device__ void row(int64_t i, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3* o3, const float* tab) const
//   Per-row scalars (angles, eps, t, ...) are read / written directly by Op::row with coalesced accesses.
//
//   Schedule of iteration k (tile = blockIdx.x + k gridDim.x, stage = k & 1), see so3d_tma.cuh:
//     wait full[stage]  ->  every thread copies its row to registers  ->  barrier A (the stage may be refilled;
//     thread 0 has drained the bulk store issued two iterations ago)  ->  thread 0 issues the bulk loads of
//     tile k+2 into `stage`  ->  Op::row  ->  results to out[stage]  ->  proxy fence + barrier B  ->
//     thread 0 issues the bulk stores of out[stage].
//   A tile that is not a full tile of 16-byte aligned arrays (ragged tail, unaligned views) is moved
//   cooperatively with ordinary loads/stores at the same points of the schedule.
// ------------------------------------------------------------------------------------------------
template <int W>
__device__ __forceinline__ void coop_load(float* __restrict__ sm, const float* __restrict__ g, int rows) {
  for (int i = threadIdx.x; i < rows * W; i += kTile) sm[i] = __ldcs(g + i);
}
template <int W>
__device__ __forceinline__ void coop_store(float* __restrict__ g, const float* __restrict__ sm, int rows) {
  for (int i = threadIdx.x; i < rows * W; i += kTile) __stcs(g + i, sm[i]);
}

__device__ __forceinline__ Mat3 sm_mat(const float* sm, int r) {
  Mat3 m;
#pragma unroll
  for (int k = 0; k < 9; ++k) m.m[k] = sm[r * 9 + k];
  return m;
}
__device__ __forceinline__ void sm_put_mat(float* sm, int r, const Mat3& m) {
#pragma unroll
  for (int k = 0; k < 9; ++k) sm[r * 9 + k] = m.m[k];
}
__device__ __forceinline__ Vec3 sm_vec(const float* sm, int r) { return Vec3{sm[r * 3], sm[r * 3 + 1], sm[r * 3 + 2]}; }
__device__ __forceinline__ void sm_put_vec(float* sm, int r, Vec3 v) {
  sm[r * 3] = v.x;
  sm[r * 3 + 1] = v.y;
  sm[r * 3 + 2] = v.z;
}

// Optional software pipeline for per-row scalars and table look-ups (latency-bound ops): an Op may define
//   struct Pre1; struct Pre2;
//   __device__ Pre1 prefetch1(int64_t i) const;               -- issued two tiles ahead (e.g. t[i], eps[i])
//   __device__ Pre2 prefetch2(int64_t i, const Pre1&) const;  -- issued one tile ahead (loads that depend on Pre1)
//   __device__ void row(int64_t i, const Pre2&, a9, a3, o9, o3, tab) const;
// so that by the time a row is processed its dependent global/L2 loads have had a whole tile time to land.
template <class Op, class = void>
struct HasPre : std::false_type {};
template <class Op>
struct HasPre<Op, std::void_t<typename Op::Pre1, typename Op::Pre2>> : std::true_type {};
struct NoPre {};
template <class Op, bool = HasPre<Op>::value>
struct PreTypes {
  using P1 = NoPre;
  using P2 = NoPre;
};
template <class Op>
struct PreTypes<Op, true> {
  using P1 = typename Op::Pre1;
  using P2 = typename Op::Pre2;
};

template <class Op>
struct OpLayout {
  static constexpr int kInWords = Op::kIn9 * 9 + Op::kIn3 * 3;     // per row
  static constexpr int kOutWords = Op::kOut9 * 9 + Op::kOut3 * 3;  // per row
  static constexpr int kOutStages = Op::kOutStages;               // 2: output tile double-buffered; 1: single (more CTAs/SM)
  static constexpr int kInFloats = kTile * kInWords;              // per stage
  static constexpr int kOutFloats = kTile * kOutWords;            // per stage
  static constexpr int kTabFloats = (Op::kTab + 3) & ~3;
  static constexpr size_t kSmemBytes = sizeof(float) * (size_t)(2 * kInFloats + kOutStages * kOutFloats + kTabFloats) + 2 * sizeof(uint64_t) + 2 * sizeof(uint32_t);
};

// register cap per op: minimum resident CTAs per SM promised to the compiler (0 = no cap)
template <class Op, class = void>
struct OpMinCtas {
  static constexpr int value = 1;
};
template <class Op>
struct OpMinCtas<Op, std::void_t<decltype(Op::kMinCtas)>> {
  static constexpr int value = Op::kMinCtas;
};

// schedule per op: ops whose rows chase per-row table entries through L2 (latency spread between warps) run the
// warp-autonomous schedule below; streaming ops keep the CTA-synchronous one (fewer per-warp issue slots).
// Measured on B200, 2^24 rows (profiles/r01k_probe_engine.jsonl): forward noising 0.577 -> 0.480 ms, per-row-t
// reverse step 0.522 -> 0.475 ms with the warp schedule; closed-form score 0.191 -> 0.212 ms, log 0.213 -> 0.235 ms
// (the per-warp store issue costs more than the barriers did), so those stay CTA-synchronous.
template <class Op, class = void>
struct OpWarpSchedule {
  static constexpr bool value = false;
};
template <class Op>
struct OpWarpSchedule<Op, std::void_t<decltype(Op::kWarpSchedule)>> {
  static constexpr bool value = Op::kWarpSchedule;
};

// An op may set Op::kWideIndex to keep the 64-bit per-tile index arithmetic of the first engine.  The tile loop is
// noise for the compute-bound series kernel, but ptxas's list schedule of its unrolled block is sensitive to the
// surrounding code: with the 32-term source form the strength-reduced indices below made the SAME instructions come
// out in an order that ran 2.6 % slower (11.29 vs 11.00 ms per 2^24 evaluations, profiles/r01x_bench.json vs r01q);
// with the shipped 64-term form it is the other way round (10.60 vs 10.70 ms), so the knob is now off
// (SO3D_SERIES_WIDE_INDEX).
template <class Op, class = void>
struct OpWideIndex {
  static constexpr bool value = false;
};
template <class Op>
struct OpWideIndex<Op, std::void_t<decltype(Op::kWideIndex)>> {
  static constexpr bool value = Op::kWideIndex;
};

template <class Op>
__global__ void __launch_bounds__(kTile, OpMinCtas<Op>::value) rowwise_kernel_cta(const Op op, const int64_t n, const int use_tma) {
  extern __shared__ float4 smem4[];
  constexpr int kI9 = Op::kIn9, kI3 = Op::kIn3, kO9 = Op::kOut9, kO3 = Op::kOut3;
  using Lay = OpLayout<Op>;
  float* smem = reinterpret_cast<float*>(smem4);
  // [in stage 0][in stage 1][out stage 0][out stage 1 if double-buffered]; every array starts 16-byte aligned
  float* s_out = smem + 2 * Lay::kInFloats;
  float* s_tab = s_out + Lay::kOutStages * Lay::kOutFloats;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_tab + Lay::kTabFloats);
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_barrier_init();
  }
  __syncthreads();  // barrier objects exist for every thread (and for compute-sanitizer's racecheck, which otherwise
                    // reports thread 0's own init -> expect_tx sequence as a hazard); costs nothing at kernel start

  // Tile k of this CTA starts at row first_row + k stride_rows.  Only the globally last tile can be ragged, and it is
  // the last tile of the CTA that owns it, so "tile k is full" is the 32-bit test k < my_full and the row index is
  // carried incrementally: no 64-bit multiplies in the tile loop (the kernels are issue-bound, DESIGN.md 4.3).
  constexpr bool kWide = OpWideIndex<Op>::value;
  using KIdx = std::conditional_t<kWide, int64_t, int>;
  const int64_t tiles = (n + kTile - 1) / kTile;
  const KIdx my_tiles = (tiles > (int64_t)blockIdx.x) ? (KIdx)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  const int my_full = (int)my_tiles - (((n % kTile) != 0 && (tiles - 1) % gridDim.x == blockIdx.x) ? 1 : 0);
  const int64_t first_row = (int64_t)blockIdx.x * kTile, stride_rows = (int64_t)gridDim.x * kTile;
  auto tile_row0 = [&](KIdx k) -> int64_t {  // off the per-tile path unless kWide
    if constexpr (kWide) return (blockIdx.x + k * gridDim.x) * (int64_t)kTile;
    else return first_row + k * stride_rows;
  };
  auto tile_rows = [&](KIdx k, int64_t row0) -> int {
    if constexpr (kWide) {
      const int64_t left = n - row0;
      return (int)(left < kTile ? left : kTile);
    } else {
      return k < my_full ? kTile : (int)(n - row0);
    }
  };
  auto tile_full = [&](KIdx k) -> bool {  // tile k exists and is a full tile
    if constexpr (kWide) return k < my_tiles && tile_rows(k, tile_row0(k)) == kTile;
    else return k < my_full;
  };
  auto issue_load = [&](KIdx k, int64_t row0) {  // thread 0 only
    if (kI9 + kI3 == 0) return;
    const int st = (int)(k & 1);
    float* base = smem + st * Lay::kInFloats;
    mbar_expect_tx(&bars[st], (uint32_t)(kTile * Lay::kInWords * sizeof(float)));
#pragma unroll
    for (int a = 0; a < kI9; ++a) bulk_load(base + a * kTile * 9, op.in9[a] + row0 * 9, kTile * 9 * sizeof(float), &bars[st]);
#pragma unroll
    for (int a = 0; a < kI3; ++a) bulk_load(base + kI9 * kTile * 9 + a * kTile * 3, op.in3[a] + row0 * 3, kTile * 3 * sizeof(float), &bars[st]);
  };
  // the first two tiles are requested BEFORE the op stages its tables, so their DRAM latency overlaps the setup
  // (thread 0 initialised the barriers itself; the other threads first touch them after the __syncthreads below)
  if (tid == 0 && use_tma) {
    if (tile_full(0)) issue_load(0, tile_row0(0));
    if (tile_full(1)) issue_load(1, tile_row0(1));
  }
  op.setup(s_tab);
  __syncthreads();

  // software pipeline registers (empty structs for ops without prefetch hooks)
  constexpr bool kPre = HasPre<Op>::value;
  typename PreTypes<Op>::P1 p1_next{};   // Pre1 of tile k+1
  typename PreTypes<Op>::P2 p2_cur{};    // Pre2 of tile k
  auto pre_row = [&](int64_t row0) -> int64_t {  // this thread's row of the tile at row0, clamped into range (result unused if beyond)
    const int64_t i = row0 + tid;
    return i < n ? i : n - 1;
  };
  if constexpr (kPre) {
    if (my_tiles > 0) p2_cur = op.prefetch2(pre_row(first_row), op.prefetch1(pre_row(first_row)));
    if (my_tiles > 1) p1_next = op.prefetch1(pre_row(first_row + stride_rows));
  }

  int64_t row_run = first_row;
  for (KIdx k = 0; k < my_tiles; ++k, row_run += stride_rows) {
    const int st = (int)(k & 1);
    const int64_t row0 = kWide ? tile_row0(k) : row_run;
    const int rows = tile_rows(k, row0);
    const bool tma = use_tma && rows == kTile;
    float* s_i9 = smem + st * Lay::kInFloats;
    float* s_i3 = s_i9 + kI9 * kTile * 9;
    float* s_o9 = s_out + (Lay::kOutStages == 2 ? st : 0) * Lay::kOutFloats;
    float* s_o3 = s_o9 + kO9 * kTile * 9;
    if (kI9 + kI3 > 0) {
      if (tma) {
        mbar_wait(&bars[st], (uint32_t)((k >> 1) & 1));
      } else {
#pragma unroll
        for (int a = 0; a < kI9; ++a) coop_load<9>(s_i9 + a * kTile * 9, op.in9[a] + row0 * 9, rows);
#pragma unroll
        for (int a = 0; a < kI3; ++a) coop_load<3>(s_i3 + a * kTile * 3, op.in3[a] + row0 * 3, rows);
        __syncthreads();
      }
    }
    Mat3 a9[kI9 > 0 ? kI9 : 1];
    Vec3 a3[kI3 > 0 ? kI3 : 1];
#pragma unroll
    for (int a = 0; a < kI9; ++a) a9[a] = sm_mat(s_i9 + a * kTile * 9, tid);
#pragma unroll
    for (int a = 0; a < kI3; ++a) a3[a] = sm_vec(s_i3 + a * kTile * 3, tid);
    if (Lay::kOutStages == 2 && tid == 0) bulk_wait_read<1>();  // the stores that read out[st] two iterations ago have drained
    __syncthreads();                                            // A
    if (tid == 0 && use_tma && tile_full(k + 2)) issue_load(k + 2, kWide ? tile_row0(k + 2) : row0 + 2 * stride_rows);

    Mat3 o9[kO9 > 0 ? kO9 : 1];
    Vec3 o3[kO3 > 0 ? kO3 : 1];
    if constexpr (kPre) {
      typename PreTypes<Op>::P2 p2_next{};
      typename PreTypes<Op>::P1 p1_next2{};
      if (k + 1 < my_tiles) p2_next = op.prefetch2(pre_row(row0 + stride_rows), p1_next);  // loads land during this tile's arithmetic
      if (k + 2 < my_tiles) p1_next2 = op.prefetch1(pre_row(row0 + 2 * stride_rows));
      if (tid < rows) op.row(row0 + tid, p2_cur, a9, a3, o9, o3, s_tab);
      p2_cur = p2_next;
      p1_next = p1_next2;
    } else {
      if (tid < rows) op.row(row0 + tid, a9, a3, o9, o3, s_tab);
    }
    if (Lay::kOutStages == 1 && kO9 + kO3 > 0) {
      // single output stage: the previous tile's stores had the whole arithmetic phase to drain
      if (tid == 0) bulk_wait_read<0>();
      __syncthreads();  // C
    }
    if (tid < rows) {
#pragma unroll
      for (int a = 0; a < kO9; ++a) sm_put_mat(s_o9 + a * kTile * 9, tid, o9[a]);
#pragma unroll
      for (int a = 0; a < kO3; ++a) sm_put_vec(s_o3 + a * kTile * 3, tid, o3[a]);
    }
    if (kO9 + kO3 > 0) {
      if (tma) {
        fence_proxy_async();
        __syncthreads();  // B
        if (tid == 0) {
#pragma unroll
          for (int a = 0; a < kO9; ++a)
            if (op.out9[a]) bulk_store(op.out9[a] + row0 * 9, s_o9 + a * kTile * 9, kTile * 9 * sizeof(float));
#pragma unroll
          for (int a = 0; a < kO3; ++a)
            if (op.out3[a]) bulk_store(op.out3[a] + row0 * 3, s_o3 + a * kTile * 3, kTile * 3 * sizeof(float));
          bulk_commit();
        }
      } else {
        __syncthreads();  // B
#pragma unroll
        for (int a = 0; a < kO9; ++a)
          if (op.out9[a]) coop_store<9>(op.out9[a] + row0 * 9, s_o9 + a * kTile * 9, rows);
#pragma unroll
        for (int a = 0; a < kO3; ++a)
          if (op.out3[a]) coop_store<3>(op.out3[a] + row0 * 3, s_o3 + a * kTile * 3, rows);
      }
    }
  }
  if (tid == 0) bulk_wait_read<0>();
}

// Warp-autonomous schedule (no CTA-wide barrier inside the tile loop):
//   * input: one bulk load per array and 256-row tile into stage k & 1, completion on full[stage]; every warp
//     waits on the mbarrier itself, copies its 32 rows to registers and releases the stage by an acq_rel
//     atomic add on a per-stage counter -- the LAST warp to release (old & 7 == 7) issues the bulk loads of
//     tile k+2 into the stage it has just freed, so nobody ever waits for a producer;
//   * output: each warp owns the 32-row slice [32 w, 32 w + 32) of the output stage (32 x 36 B = 1152 B,
//     32 x 12 B = 384 B: contiguous, 16-byte aligned), fences it to the async proxy and lane 0 issues the
//     warp's own bulk stores; the warp's bulk groups are drained by lane 0 before the slice is reused;
//   * ragged tail / unaligned arrays: the warp moves its own rows with coalesced ld/st.global.cs.
// Warps of a CTA drift freely (by up to two tiles), which hides the per-row latency spread of the table
// look-ups and removes the barrier stalls of the CTA-synchronous schedule (ncu r01e: 1.4-4.4 stalled warps
// per issue on the reverse step / forward noising kernels).
template <int W>
__device__ __forceinline__ void warp_load(float* __restrict__ sm, const float* __restrict__ g, int rows, int lane) {
  for (int i = lane; i < rows * W; i += 32) sm[i] = __ldcs(g + i);
}
template <int W>
__device__ __forceinline__ void warp_store(float* __restrict__ g, const float* __restrict__ sm, int rows, int lane) {
  for (int i = lane; i < rows * W; i += 32) __stcs(g + i, sm[i]);
}
__device__ __forceinline__ uint32_t atom_add_acq_rel_cta(uint32_t* p, uint32_t v) {
  uint32_t old;
  asm volatile("atom.acq_rel.cta.shared::cta.add.u32 %0, [%1], %2;" : "=r"(old) : "r"(smem_u32(p)), "r"(v) : "memory");
  return old;
}

__device__ __forceinline__ bool elect_one() {  // one lane of the (converged) warp
  uint32_t pred;
  asm volatile("{\n .reg .pred p;\n elect.sync _|p, 0xffffffff;\n selp.u32 %0, 1, 0, p;\n}\n" : "=r"(pred));
  return pred != 0;
}

template <class Op>
__global__ void __launch_bounds__(kTile, OpMinCtas<Op>::value) rowwise_kernel(const Op op, const int64_t n, const int use_tma) {
  extern __shared__ float4 smem4[];
  constexpr int kI9 = Op::kIn9, kI3 = Op::kIn3, kO9 = Op::kOut9, kO3 = Op::kOut3;
  constexpr int kWarps = kTile / 32;
  using Lay = OpLayout<Op>;
  float* smem = reinterpret_cast<float*>(smem4);
  // [in stage 0][in stage 1][out stage 0][out stage 1 if double-buffered]; every array starts 16-byte aligned
  float* s_out = smem + 2 * Lay::kInFloats;
  float* s_tab = s_out + Lay::kOutStages * Lay::kOutFloats;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_tab + Lay::kTabFloats);
  uint32_t* released = reinterpret_cast<uint32_t*>(bars + 2);  // per input stage: warps that have copied their rows out
  const int tid = threadIdx.x, lane = tid & 31;
#if SO3D_WROW_SHFL
  // a broadcast from lane 0 tells the compiler the value is warp-uniform: the bulk-copy operands (uniform registers in
  // SASS) then need one R2UR each instead of a predicate waterfall loop per copy (24 -> ~8 issue slots per copy, r03u)
  const int wrow = __shfl_sync(0xffffffffu, tid & ~31, 0);
#else
  const int wrow = tid & ~31;
#endif
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    released[0] = 0;
    released[1] = 0;
    fence_barrier_init();
  }
  __syncthreads();  // see rowwise_kernel_cta

  // Tile k of this CTA starts at row first_row + k stride_rows.  Only the globally last tile can be ragged, and it is
  // the last tile of the CTA that owns it, so "tile k is full" is the 32-bit test k < my_full and the row index is
  // carried incrementally: no 64-bit multiplies in the tile loop (the kernels are issue-bound, DESIGN.md 4.3).
  const int64_t tiles = (n + kTile - 1) / kTile;
  const int my_tiles = (tiles > (int64_t)blockIdx.x) ? (int)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  const int my_full = my_tiles - (((n % kTile) != 0 && (tiles - 1) % gridDim.x == blockIdx.x) ? 1 : 0);
  const int64_t first_row = (int64_t)blockIdx.x * kTile, stride_rows = (int64_t)gridDim.x * kTile;
  auto tile_row0 = [&](int k) -> int64_t { return first_row + k * stride_rows; };  // off the per-tile path
  auto issue_load = [&](int k, int64_t row0) {  // one thread
    if (kI9 + kI3 == 0) return;
    const int st = k & 1;
    float* base = smem + st * Lay::kInFloats;
    mbar_expect_tx(&bars[st], (uint32_t)(kTile * Lay::kInWords * sizeof(float)));
#pragma unroll
    for (int a = 0; a < kI9; ++a) bulk_load(base + a * kTile * 9, op.in9[a] + row0 * 9, kTile * 9 * sizeof(float), &bars[st]);
#pragma unroll
    for (int a = 0; a < kI3; ++a) bulk_load(base + kI9 * kTile * 9 + a * kTile * 3, op.in3[a] + row0 * 3, kTile * 3 * sizeof(float), &bars[st]);
  };
  if (tid == 0 && use_tma) {  // before the op's setup: the first tiles' DRAM latency overlaps the table staging
    if (my_full > 0) issue_load(0, tile_row0(0));
    if (my_full > 1) issue_load(1, tile_row0(1));
  }
  op.setup(s_tab);
  __syncthreads();

  // software pipeline registers (empty structs for ops without prefetch hooks)
  constexpr bool kPre = HasPre<Op>::value;
  typename PreTypes<Op>::P1 p1_next{};   // Pre1 of tile k+1
  typename PreTypes<Op>::P2 p2_cur{};    // Pre2 of tile k
  auto pre_row = [&](int64_t row0) -> int64_t {  // this thread's row of the tile at row0, clamped into range (result unused if beyond)
    const int64_t i = row0 + tid;
    return i < n ? i : n - 1;
  };
  if constexpr (kPre) {
    if (my_tiles > 0) p2_cur = op.prefetch2(pre_row(first_row), op.prefetch1(pre_row(first_row)));
    if (my_tiles > 1) p1_next = op.prefetch1(pre_row(first_row + stride_rows));
  }

  int64_t row0 = first_row;
  for (int k = 0; k < my_tiles; ++k, row0 += stride_rows) {
    const int st = k & 1;
    const int rows = k < my_full ? kTile : (int)(n - row0);
    const bool tma = use_tma && rows == kTile;
    int wrows = rows - wrow;  // rows of this warp's slice that exist
    wrows = wrows < 0 ? 0 : (wrows > 32 ? 32 : wrows);
    float* s_i9 = smem + st * Lay::kInFloats;
    float* s_i3 = s_i9 + kI9 * kTile * 9;
    float* s_o9 = s_out + (Lay::kOutStages == 2 ? st : 0) * Lay::kOutFloats;
    float* s_o3 = s_o9 + kO9 * kTile * 9;
    if (kI9 + kI3 > 0) {
      if (tma) {
        mbar_wait(&bars[st], (uint32_t)((k >> 1) & 1));
      } else {
#pragma unroll
        for (int a = 0; a < kI9; ++a) warp_load<9>(s_i9 + a * kTile * 9 + wrow * 9, op.in9[a] + (row0 + wrow) * 9, wrows, lane);
#pragma unroll
        for (int a = 0; a < kI3; ++a) warp_load<3>(s_i3 + a * kTile * 3 + wrow * 3, op.in3[a] + (row0 + wrow) * 3, wrows, lane);
        __syncwarp();
      }
    }
    Mat3 a9[kI9 > 0 ? kI9 : 1];
    Vec3 a3[kI3 > 0 ? kI3 : 1];
#pragma unroll
    for (int a = 0; a < kI9; ++a) a9[a] = sm_mat(s_i9 + a * kTile * 9, tid);
#pragma unroll
    for (int a = 0; a < kI3; ++a) a3[a] = sm_vec(s_i3 + a * kTile * 3, tid);
    if (kI9 + kI3 > 0) {
      __syncwarp();  // every lane's copy of its row is complete
      if (tma && lane == 0 && k + 2 < my_full) {
        const uint32_t old = atom_add_acq_rel_cta(&released[st], 1u);
        if ((old & (kWarps - 1)) == kWarps - 1) issue_load(k + 2, row0 + 2 * stride_rows);  // last warp out refills the stage
      }
    }

    Mat3 o9[kO9 > 0 ? kO9 : 1];
    Vec3 o3[kO3 > 0 ? kO3 : 1];
    if constexpr (kPre) {
      typename PreTypes<Op>::P2 p2_next{};
      typename PreTypes<Op>::P1 p1_next2{};
      if (k + 1 < my_tiles) p2_next = op.prefetch2(pre_row(row0 + stride_rows), p1_next);  // loads land during this tile's arithmetic
      if (k + 2 < my_tiles) p1_next2 = op.prefetch1(pre_row(row0 + 2 * stride_rows));
      if (tid < rows) op.row(row0 + tid, p2_cur, a9, a3, o9, o3, s_tab);
      p2_cur = p2_next;
      p1_next = p1_next2;
    } else {
      if (tid < rows) op.row(row0 + tid, a9, a3, o9, o3, s_tab);
    }
    if (kO9 + kO3 > 0) {
      // this warp's earlier bulk stores must have finished reading the slice that is about to be overwritten.  Bulk
      // groups belong to the thread that committed them; every lane waits (lanes without groups fall through), so
      // the wait does not depend on which lane elect.sync picked for the store issue
      if (SO3D_WROW_SHFL || lane == 0) {
        if (Lay::kOutStages == 2) bulk_wait_read<1>(); else bulk_wait_read<0>();
      }
      __syncwarp();
      if (tid < rows) {
#pragma unroll
        for (int a = 0; a < kO9; ++a) sm_put_mat(s_o9 + a * kTile * 9, tid, o9[a]);
#pragma unroll
        for (int a = 0; a < kO3; ++a) sm_put_vec(s_o3 + a * kTile * 3, tid, o3[a]);
      }
      if (tma) {
        fence_proxy_async();
        __syncwarp();
        if (SO3D_WROW_SHFL ? elect_one() : lane == 0) {
#pragma unroll
          for (int a = 0; a < kO9; ++a)
            if (op.out9[a]) bulk_store(op.out9[a] + (row0 + wrow) * 9, s_o9 + a * kTile * 9 + wrow * 9, 32 * 9 * sizeof(float));
#pragma unroll
          for (int a = 0; a < kO3; ++a)
            if (op.out3[a]) bulk_store(op.out3[a] + (row0 + wrow) * 3, s_o3 + a * kTile * 3 + wrow * 3, 32 * 3 * sizeof(float));
          bulk_commit();
        }
      } else {
        __syncwarp();
#pragma unroll
        for (int a = 0; a < kO9; ++a)
          if (op.out9[a]) warp_store<9>(op.out9[a] + (row0 + wrow) * 9, s_o9 + a * kTile * 9 + wrow * 9, wrows, lane);
#pragma unroll
        for (int a = 0; a < kO3; ++a)
          if (op.out3[a]) warp_store<3>(op.out3[a] + (row0 + wrow) * 3, s_o3 + a * kTile * 3 + wrow * 3, wrows, lane);
        __syncwarp();  // the slice may be rewritten next iteration (single output stage)
      }
    }
  }
  if (SO3D_WROW_SHFL || lane == 0) bulk_wait_read<0>();
}

template <class Op>
int launch_rowwise(const Op& op, int64_t n, void* stream, const char* name, int ctas_per_sm = 0) {
  if (n < 0) return fail(SO3D_EINVAL, "negative n");
  if (n == 0) return 0;
  int use_tma = 1;
  for (int a = 0; a < Op::kIn9; ++a) {
    if (!op.in9[a]) return fail(SO3D_EINVAL, "null input pointer");
    use_tma &= aligned16(op.in9[a]);
  }
  for (int a = 0; a < Op::kIn3; ++a) {
    if (!op.in3[a]) return fail(SO3D_EINVAL, "null input pointer");
    use_tma &= aligned16(op.in3[a]);
  }
  for (int a = 0; a < Op::kOut9; ++a) use_tma &= aligned16(op.out9[a]);
  for (int a = 0; a < Op::kOut3; ++a) use_tma &= aligned16(op.out3[a]);
  constexpr size_t smem = OpLayout<Op>::kSmemBytes;
  static_assert(smem <= 227 * 1024, "tile stages exceed shared memory");
  // Persistent grid = exactly the CTAs that are resident at once (registers and shared memory both count): with
  // a static partition of the tiles, a grid larger than one wave leaves the last, partial wave's SMs idle.
  static int resident_dev[2][kMaxDevices] = {};  // per Op instantiation, schedule and device
  int* resident = nullptr;
  static const int cta_sync = [] {  // A/B aid: SO3D_ENGINE=cta|warp overrides the op's own choice
    const char* e = getenv("SO3D_ENGINE");
    if (e && strcmp(e, "cta") == 0) return 1;
    if (e && strcmp(e, "warp") == 0) return 0;
    return OpWarpSchedule<Op>::value ? 0 : 1;
  }();
  auto kern = cta_sync ? rowwise_kernel_cta<Op> : rowwise_kernel<Op>;
  const int dev = current_device();
  int per_schedule[2] = {resident_dev[0][dev], resident_dev[1][dev]};
  resident = per_schedule;
  if (resident[cta_sync] == 0) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kTile, smem) != cudaSuccess || occ < 1) occ = 1;
    resident[cta_sync] = occ;
    resident_dev[cta_sync][dev] = occ;
  }
  if (ctas_per_sm <= 0 || ctas_per_sm > resident[cta_sync]) ctas_per_sm = resident[cta_sync];
  if (const char* e = getenv("SO3D_CTAS_PER_SM")) {  // tuning aid: cap the persistent grid (CTAs per SM)
    const int v = atoi(e);
    if (v > 0 && v < ctas_per_sm) ctas_per_sm = v;
  }
  kern<<<grid_for(n, ctas_per_sm), kTile, smem, (cudaStream_t)stream>>>(op, n, use_tma);
  return check_launch(name);
}

// ------------------------------------------------------------------------------------------------
// Two rows per thread (so3d_lanes.cuh).  The same two schedules with tiles of 2 x kTile = 512 rows moved by 256 threads:
// thread `tid` owns rows `tid` and `tid + 256` of a tile and carries them through the op's arithmetic as the two lanes of
// packed FP32 instructions (FFMA2 / FMUL2 / FADD2): half the issue slots for the ~45 % of a fused step that is FP32
// arithmetic.  These are separate kernel templates, not a parameter of the ones above: the one-row kernels' code
// (and with it ptxas's schedule of the compute-bound series kernel) stays exactly as it was.
//   Op2 provides kIn9 / kIn3 / kOut9 / kOut3 / kOutStages / kTab / setup() like a one-row op, and
//     __device__ void row2(int64_t i0, const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*o3)[2], const float* tab) const
//   for the rows i0 (lane 0) and i0 + kTile (lane 1); a lane beyond the end of the data computes on stale values and its
//   results are dropped.
// ------------------------------------------------------------------------------------------------
#ifndef SO3D_LANES2_THREADS
#define SO3D_LANES2_THREADS 128  // threads per CTA of the two-row kernels: 128 -> 256-row tiles like the one-row kernels (same shared
#endif                           // memory per CTA, 4 resident CTAs of 4 warps); 256 -> 512-row tiles, 2 resident CTAs of 8 warps
constexpr int kT2 = SO3D_LANES2_THREADS;  // thread `tid` owns rows `tid` and `tid + kT2` of a tile
constexpr int kRows2 = 2 * kT2;
template <int W>
__device__ __forceinline__ void coop_load2(float* __restrict__ sm, const float* __restrict__ g, int rows) {
  for (int i = threadIdx.x; i < rows * W; i += kT2) sm[i] = __ldcs(g + i);
}
template <int W>
__device__ __forceinline__ void coop_store2(float* __restrict__ g, const float* __restrict__ sm, int rows) {
  for (int i = threadIdx.x; i < rows * W; i += kT2) __stcs(g + i, sm[i]);
}

// input stages of a two-row op: 2 (tile k+2 in flight while k is computed) or 1 (the single stage is refilled with tile
// k+1 as soon as every thread holds its rows of tile k in registers: 12 KB less shared memory per CTA -> more resident CTAs)
template <class Op, class = void>
struct OpInStages {
  static constexpr int value = 2;
};
template <class Op>
struct OpInStages<Op, std::void_t<decltype(Op::kInStages)>> {
  static constexpr int value = Op::kInStages;
};

template <class Op>
struct OpLayout2 {
  static constexpr int kInWords = Op::kIn9 * 9 + Op::kIn3 * 3;
  static constexpr int kOutWords = Op::kOut9 * 9 + Op::kOut3 * 3;
  static constexpr int kOutStages = Op::kOutStages;
  static constexpr int kInFloats = kRows2 * kInWords;
  static constexpr int kOutFloats = kRows2 * kOutWords;
  static constexpr int kTabFloats = (Op::kTab + 3) & ~3;
  static constexpr int kInStages = OpInStages<Op>::value;
  static constexpr size_t kSmemBytes = sizeof(float) * (size_t)(kInStages * kInFloats + kOutStages * kOutFloats + kTabFloats) + 2 * sizeof(uint64_t) + 2 * sizeof(uint32_t);
};

template <class Op>
__global__ void __launch_bounds__(kT2, OpMinCtas<Op>::value) rowwise_kernel_cta2(const Op op, const int64_t n, const int use_tma) {
  extern __shared__ float4 smem4[];
  constexpr int kI9 = Op::kIn9, kI3 = Op::kIn3, kO9 = Op::kOut9, kO3 = Op::kOut3;
  using Lay = OpLayout2<Op>;
  float* smem = reinterpret_cast<float*>(smem4);
  constexpr int kIS = Lay::kInStages;
  float* s_out = smem + kIS * Lay::kInFloats;
  float* s_tab = s_out + Lay::kOutStages * Lay::kOutFloats;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_tab + Lay::kTabFloats);
  const int tid = threadIdx.x;
  if (tid == 0) {
    mbar_init(&bars[0], 1);
    mbar_init(&bars[1], 1);
    fence_barrier_init();
  }
  __syncthreads();
  const int64_t tiles = (n + kRows2 - 1) / kRows2;
  const int my_tiles = (tiles > (int64_t)blockIdx.x) ? (int)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  const int my_full = my_tiles - (((n % kRows2) != 0 && (tiles - 1) % gridDim.x == blockIdx.x) ? 1 : 0);
  const int64_t first_row = (int64_t)blockIdx.x * kRows2, stride_rows = (int64_t)gridDim.x * kRows2;
  auto issue_load = [&](int k, int64_t row0) {  // thread 0 only
    if (kI9 + kI3 == 0) return;
    const int st = kIS == 2 ? (k & 1) : 0;
    float* base = smem + st * Lay::kInFloats;
    mbar_expect_tx(&bars[st], (uint32_t)(kRows2 * Lay::kInWords * sizeof(float)));
#pragma unroll
    for (int a = 0; a < kI9; ++a) bulk_load(base + a * kRows2 * 9, op.in9[a] + row0 * 9, kRows2 * 9 * sizeof(float), &bars[st]);
#pragma unroll
    for (int a = 0; a < kI3; ++a) bulk_load(base + kI9 * kRows2 * 9 + a * kRows2 * 3, op.in3[a] + row0 * 3, kRows2 * 3 * sizeof(float), &bars[st]);
  };
  if (tid == 0 && use_tma) {
    if (my_full > 0) issue_load(0, first_row);
    if (kIS == 2 && my_full > 1) issue_load(1, first_row + stride_rows);
  }
  op.setup(s_tab);
  __syncthreads();

  int64_t row0 = first_row;
  for (int k = 0; k < my_tiles; ++k, row0 += stride_rows) {
    const int st = kIS == 2 ? (k & 1) : 0;
    const int rows = k < my_full ? kRows2 : (int)(n - row0);
    const bool tma = use_tma && rows == kRows2;
    float* s_i9 = smem + st * Lay::kInFloats;
    float* s_i3 = s_i9 + kI9 * kRows2 * 9;
    float* s_o9 = s_out + (Lay::kOutStages == 2 ? (k & 1) : 0) * Lay::kOutFloats;
    float* s_o3 = s_o9 + kO9 * kRows2 * 9;
    if (kI9 + kI3 > 0) {
      if (tma) {
        mbar_wait(&bars[st], (uint32_t)(kIS == 2 ? ((k >> 1) & 1) : (k & 1)));
      } else {
#pragma unroll
        for (int a = 0; a < kI9; ++a) coop_load2<9>(s_i9 + a * kRows2 * 9, op.in9[a] + row0 * 9, rows);
#pragma unroll
        for (int a = 0; a < kI3; ++a) coop_load2<3>(s_i3 + a * kRows2 * 3, op.in3[a] + row0 * 3, rows);
        __syncthreads();
      }
    }
    Mat3 a9[kI9 > 0 ? kI9 : 1][2];
    Vec3 a3[kI3 > 0 ? kI3 : 1][2];
#pragma unroll
    for (int a = 0; a < kI9; ++a) {
      a9[a][0] = sm_mat(s_i9 + a * kRows2 * 9, tid);
      a9[a][1] = sm_mat(s_i9 + a * kRows2 * 9, tid + kT2);
    }
#pragma unroll
    for (int a = 0; a < kI3; ++a) {
      a3[a][0] = sm_vec(s_i3 + a * kRows2 * 3, tid);
      a3[a][1] = sm_vec(s_i3 + a * kRows2 * 3, tid + kT2);
    }
    if (Lay::kOutStages == 2 && tid == 0) bulk_wait_read<1>();
    __syncthreads();  // A
    if (tid == 0 && use_tma && k + kIS < my_full) issue_load(k + kIS, row0 + kIS * stride_rows);

    Mat3 o9[kO9 > 0 ? kO9 : 1][2];
    Vec3 o3[kO3 > 0 ? kO3 : 1][2];
    if (tid < rows) op.row2(row0 + tid, a9, a3, o9, o3, s_tab);
    if (Lay::kOutStages == 1 && kO9 + kO3 > 0) {
      if (tid == 0) bulk_wait_read<0>();
      __syncthreads();  // C
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      if (tid + j * kT2 < rows) {
#pragma unroll
        for (int a = 0; a < kO9; ++a) sm_put_mat(s_o9 + a * kRows2 * 9, tid + j * kT2, o9[a][j]);
#pragma unroll
        for (int a = 0; a < kO3; ++a) sm_put_vec(s_o3 + a * kRows2 * 3, tid + j * kT2, o3[a][j]);
      }
    }
    if (kO9 + kO3 > 0) {
      if (tma) {
        fence_proxy_async();
        __syncthreads();  // B
        if (tid == 0) {
#pragma unroll
          for (int a = 0; a < kO9; ++a)
            if (op.out9[a]) bulk_store(op.out9[a] + row0 * 9, s_o9 + a * kRows2 * 9, kRows2 * 9 * sizeof(float));
#pragma unroll
          for (int a = 0; a < kO3; ++a)
            if (op.out3[a]) bulk_store(op.out3[a] + row0 * 3, s_o3 + a * kRows2 * 3, kRows2 * 3 * sizeof(float));
          bulk_commit();
        }
      } else {
        __syncthreads();  // B
#pragma unroll
        for (int a = 0; a < kO9; ++a)
          if (op.out9[a]) coop_store2<9>(op.out9[a] + row0 * 9, s_o9 + a * kRows2 * 9, rows);
#pragma unroll
        for (int a = 0; a < kO3; ++a)
          if (op.out3[a]) coop_store2<3>(op.out3[a] + row0 * 3, s_o3 + a * kRows2 * 3, rows);
      }
    }
  }
  if (tid == 0) bulk_wait_read<0>();
}

template <class Op>
int launch_rowwise2(const Op& op, int64_t n, void* stream, const char* name) {
  if (n < 0) return fail(SO3D_EINVAL, "negative n");
  if (n == 0) return 0;
  int use_tma = 1;
  for (int a = 0; a < Op::kIn9; ++a) {
    if (!op.in9[a]) return fail(SO3D_EINVAL, "null input pointer");
    use_tma &= aligned16(op.in9[a]);
  }
  for (int a = 0; a < Op::kIn3; ++a) {
    if (!op.in3[a]) return fail(SO3D_EINVAL, "null input pointer");
    use_tma &= aligned16(op.in3[a]);
  }
  for (int a = 0; a < Op::kOut9; ++a) use_tma &= aligned16(op.out9[a]);
  for (int a = 0; a < Op::kOut3; ++a) use_tma &= aligned16(op.out3[a]);
  constexpr size_t smem = OpLayout2<Op>::kSmemBytes;
  static_assert(smem <= 227 * 1024, "tile stages exceed shared memory");
  static int resident_dev[kMaxDevices] = {};
  auto kern = rowwise_kernel_cta2<Op>;
  const int dev = current_device();
  if (resident_dev[dev] == 0) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kT2, smem) != cudaSuccess || occ < 1) occ = 1;
    resident_dev[dev] = occ;
  }
  int ctas_per_sm = resident_dev[dev];
  if (const char* e = getenv("SO3D_CTAS_PER_SM")) {
    const int v = atoi(e);
    if (v > 0 && v < ctas_per_sm) ctas_per_sm = v;
  }
  const int64_t tiles = (n + kRows2 - 1) / kRows2;
  const int64_t cap = (int64_t)sm_count() * ctas_per_sm;
  kern<<<(int)(tiles < cap ? tiles : cap), kT2, smem, (cudaStream_t)stream>>>(op, n, use_tma);
  return check_launch(name);
}

// ------------------------------------------------------------------------------------------------
// Two rows per thread on the WARP-AUTONOMOUS schedule (rowwise_kernel_w2): for the latency-spread ops that also define
// prefetch hooks.  A CTA of kT2 threads moves tiles of kRows2 = 2 kT2 rows; warp w owns the 64 consecutive rows
// [64 w, 64 w + 64) of a tile, thread `lane` of it the rows 64 w + lane (lane 0 of the packed arithmetic) and
// 64 w + 32 + lane (lane 1).  Input side as in rowwise_kernel (CTA-wide bulk loads into a two-stage ring, the last warp
// that has copied its rows out refills the stage); output side per warp (64-row slices: 2304 B / 768 B per array), issued
// under elect.sync.  Everything that is paid once per warp and tile -- ring wait, stage release, fence, store issue, tile
// bookkeeping -- is paid per 64 rows instead of per 32, and the op's FP32 arithmetic runs as FFMA2 / FMUL2 / FADD2.
//   Op2 provides Pre1 / Pre2 / prefetch1 / prefetch2 like a one-row op (called once per row) and
//     __device__ void row2(int64_t i0, const Pre2 (&p)[2], const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*o3)[2], const float* tab) const
//   for the rows i0 (lane 0) and i0 + 32 (lane 1).
// ------------------------------------------------------------------------------------------------
// An op may set Op::kBranchless: no branches around the prefetch of the next tiles and the rows' arithmetic, so that ptxas
// schedules the integer-heavy prefetch (Philox, address arithmetic) and the FP32 arithmetic of the current rows as ONE block.
// Row indices are clamped to n - 1, so a prefetch beyond the CTA's last tile re-reads valid entries; rows beyond the end of
// a ragged tile compute on stale shared memory and are not stored.  Measured per op (r04c): forward noising with the score
// 0.393 -> 0.385 ms, plain forward noising 0.323 -> 0.365 ms (a 96-register schedule that overlaps less) -- hence a trait.
template <class Op, class = void>
struct OpBranchless {
  static constexpr bool value = false;
};
template <class Op>
struct OpBranchless<Op, std::void_t<decltype(Op::kBranchless)>> {
  static constexpr bool value = Op::kBranchless;
};
template <class Op>
__global__ void __launch_bounds__(kT2, OpMinCtas<Op>::value) rowwise_kernel_w2(const Op op, const int64_t n, const int use_tma) {
  extern __shared__ float4 smem4[];
  constexpr int kI9 = Op::kIn9, kI3 = Op::kIn3, kO9 = Op::kOut9, kO3 = Op::kOut3;
  constexpr int kWarps = kT2 / 32;
  using Lay = OpLayout2<Op>;
  // kWarpIn (Op::kInStages == 1): ONE input stage, every warp loads its own 64-row slice (its own mbarrier) and refills it as
  // soon as its rows are in registers -- no ring, no release counter, no coupling between the warps of a CTA, and 12 KB
  // less shared memory.  Otherwise (two stages): CTA-wide loads into a ring, the last warp out refills the stage.
  constexpr bool kWarpIn = Lay::kInStages == 1;
  float* smem = reinterpret_cast<float*>(smem4);
  float* s_out = smem + Lay::kInStages * Lay::kInFloats;
  float* s_tab = s_out + Lay::kOutStages * Lay::kOutFloats;
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_tab + Lay::kTabFloats);  // kWarpIn: one per warp;  else two + the release counters
  uint32_t* released = reinterpret_cast<uint32_t*>(bars + 2);
  const int tid = threadIdx.x, lane = tid & 31;
  const int wrow = __shfl_sync(0xffffffffu, 2 * (tid & ~31), 0);  // first row of the warp's slice (warp-uniform: see rowwise_kernel)
  const int r0 = wrow + lane, r1 = r0 + 32;                       // this thread's two rows of a tile
  if (tid == 0) {
    if (kWarpIn) {
      for (int w = 0; w < kWarps; ++w) mbar_init(&bars[w], 1);
    } else {
      mbar_init(&bars[0], 1);
      mbar_init(&bars[1], 1);
      released[0] = 0;
      released[1] = 0;
    }
    fence_barrier_init();
  }
  __syncthreads();
  uint64_t* wbar = &bars[kWarpIn ? (wrow >> 6) : 0];  // this warp's barrier (kWarpIn)
  const int64_t tiles = (n + kRows2 - 1) / kRows2;
  const int my_tiles = (tiles > (int64_t)blockIdx.x) ? (int)((tiles - blockIdx.x + gridDim.x - 1) / gridDim.x) : 0;
  const int my_full = my_tiles - (((n % kRows2) != 0 && (tiles - 1) % gridDim.x == blockIdx.x) ? 1 : 0);
  const int64_t first_row = (int64_t)blockIdx.x * kRows2, stride_rows = (int64_t)gridDim.x * kRows2;
  auto issue_load = [&](int k, int64_t row0) {  // one thread
    if (kI9 + kI3 == 0) return;
    const int st = k & 1;
    float* base = smem + st * Lay::kInFloats;
    mbar_expect_tx(&bars[st], (uint32_t)(kRows2 * Lay::kInWords * sizeof(float)));
#pragma unroll
    for (int a = 0; a < kI9; ++a) bulk_load(base + a * kRows2 * 9, op.in9[a] + row0 * 9, kRows2 * 9 * sizeof(float), &bars[st]);
#pragma unroll
    for (int a = 0; a < kI3; ++a) bulk_load(base + kI9 * kRows2 * 9 + a * kRows2 * 3, op.in3[a] + row0 * 3, kRows2 * 3 * sizeof(float), &bars[st]);
  };
  auto issue_warp_load = [&](int64_t row0) {  // one lane: this warp's 64-row slice of the tile at row0 (kWarpIn)
    if (kI9 + kI3 == 0) return;
    mbar_expect_tx(wbar, (uint32_t)(64 * Lay::kInWords * sizeof(float)));
#pragma unroll
    for (int a = 0; a < kI9; ++a) bulk_load(smem + a * kRows2 * 9 + wrow * 9, op.in9[a] + (row0 + wrow) * 9, 64 * 9 * sizeof(float), wbar);
#pragma unroll
    for (int a = 0; a < kI3; ++a) bulk_load(smem + kI9 * kRows2 * 9 + a * kRows2 * 3 + wrow * 3, op.in3[a] + (row0 + wrow) * 3, 64 * 3 * sizeof(float), wbar);
  };
  if (kWarpIn) {
    if (use_tma && my_full > 0 && elect_one()) issue_warp_load(first_row);
  } else if (tid == 0 && use_tma) {
    if (my_full > 0) issue_load(0, first_row);
    if (my_full > 1) issue_load(1, first_row + stride_rows);
  }
  op.setup(s_tab);
  __syncthreads();

  typename Op::Pre1 p1_next[2]{};  // Pre1 of tile k+1, both rows
  typename Op::Pre2 p2_cur[2]{};   // Pre2 of tile k
  auto pre_row = [&](int64_t row0, int r) -> int64_t {  // clamped into range (the result of a row beyond the end is dropped)
    const int64_t i = row0 + r;
    return i < n ? i : n - 1;
  };
  if (my_tiles > 0) {
    p2_cur[0] = op.prefetch2(pre_row(first_row, r0), op.prefetch1(pre_row(first_row, r0)));
    p2_cur[1] = op.prefetch2(pre_row(first_row, r1), op.prefetch1(pre_row(first_row, r1)));
  }
  if (my_tiles > 1) {
    p1_next[0] = op.prefetch1(pre_row(first_row + stride_rows, r0));
    p1_next[1] = op.prefetch1(pre_row(first_row + stride_rows, r1));
  }

  int64_t row0 = first_row;
  for (int k = 0; k < my_tiles; ++k, row0 += stride_rows) {
    const int st = kWarpIn ? 0 : (k & 1);
    const int rows = k < my_full ? kRows2 : (int)(n - row0);
    const bool tma = use_tma && rows == kRows2;
    int wrows = rows - wrow;  // rows of this warp's slice that exist
    wrows = wrows < 0 ? 0 : (wrows > 64 ? 64 : wrows);
    float* s_i9 = smem + st * Lay::kInFloats;
    float* s_i3 = s_i9 + kI9 * kRows2 * 9;
    float* s_o9 = s_out + (Lay::kOutStages == 2 ? (k & 1) : 0) * Lay::kOutFloats;
    float* s_o3 = s_o9 + kO9 * kRows2 * 9;
    if (kI9 + kI3 > 0) {
      if (tma) {
        if (kWarpIn) mbar_wait(wbar, (uint32_t)(k & 1)); else mbar_wait(&bars[st], (uint32_t)((k >> 1) & 1));
      } else {
#pragma unroll
        for (int a = 0; a < kI9; ++a) warp_load<9>(s_i9 + a * kRows2 * 9 + wrow * 9, op.in9[a] + (row0 + wrow) * 9, wrows, lane);
#pragma unroll
        for (int a = 0; a < kI3; ++a) warp_load<3>(s_i3 + a * kRows2 * 3 + wrow * 3, op.in3[a] + (row0 + wrow) * 3, wrows, lane);
        __syncwarp();
      }
    }
    Mat3 a9[kI9 > 0 ? kI9 : 1][2];
    Vec3 a3[kI3 > 0 ? kI3 : 1][2];
#pragma unroll
    for (int a = 0; a < kI9; ++a) {
      a9[a][0] = sm_mat(s_i9 + a * kRows2 * 9, r0);
      a9[a][1] = sm_mat(s_i9 + a * kRows2 * 9, r1);
    }
#pragma unroll
    for (int a = 0; a < kI3; ++a) {
      a3[a][0] = sm_vec(s_i3 + a * kRows2 * 3, r0);
      a3[a][1] = sm_vec(s_i3 + a * kRows2 * 3, r1);
    }
    if (kI9 + kI3 > 0) {
      __syncwarp();  // every lane's copy of its rows is complete
      if (kWarpIn) {
        if (tma && k + 1 < my_full && elect_one()) issue_warp_load(row0 + stride_rows);  // the next tile's slice loads behind the arithmetic
      } else if (tma && lane == 0 && k + 2 < my_full) {
        const uint32_t old = atom_add_acq_rel_cta(&released[st], 1u);
        if ((old & (kWarps - 1)) == kWarps - 1) issue_load(k + 2, row0 + 2 * stride_rows);  // last warp out refills the stage
      }
    }

    Mat3 o9[kO9 > 0 ? kO9 : 1][2];
    Vec3 o3[kO3 > 0 ? kO3 : 1][2];
    {
      typename Op::Pre2 p2_next[2]{};
      typename Op::Pre1 p1_next2[2]{};
      constexpr bool kBl = OpBranchless<Op>::value;
      if (kBl || k + 1 < my_tiles) {  // loads land during this tile's arithmetic
        p2_next[0] = op.prefetch2(pre_row(row0 + stride_rows, r0), p1_next[0]);
        p2_next[1] = op.prefetch2(pre_row(row0 + stride_rows, r1), p1_next[1]);
      }
      if (kBl || k + 2 < my_tiles) {
        p1_next2[0] = op.prefetch1(pre_row(row0 + 2 * stride_rows, r0));
        p1_next2[1] = op.prefetch1(pre_row(row0 + 2 * stride_rows, r1));
      }
      if (kBl || r0 < rows) op.row2(row0 + r0, p2_cur, a9, a3, o9, o3, s_tab);
      p2_cur[0] = p2_next[0], p2_cur[1] = p2_next[1];
      p1_next[0] = p1_next2[0], p1_next[1] = p1_next2[1];
    }
    if (kO9 + kO3 > 0) {
      // every lane (see rowwise_kernel): the warp's earlier stores have finished reading the slice that is written next
      if (Lay::kOutStages == 2) bulk_wait_read<1>(); else bulk_wait_read<0>();
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        if (r0 + 32 * j < rows) {
#pragma unroll
          for (int a = 0; a < kO9; ++a) sm_put_mat(s_o9 + a * kRows2 * 9, r0 + 32 * j, o9[a][j]);
#pragma unroll
          for (int a = 0; a < kO3; ++a) sm_put_vec(s_o3 + a * kRows2 * 3, r0 + 32 * j, o3[a][j]);
        }
      }
      if (tma) {
        fence_proxy_async();
        __syncwarp();
        if (elect_one()) {
#pragma unroll
          for (int a = 0; a < kO9; ++a)
            if (op.out9[a]) bulk_store(op.out9[a] + (row0 + wrow) * 9, s_o9 + a * kRows2 * 9 + wrow * 9, 64 * 9 * sizeof(float));
#pragma unroll
          for (int a = 0; a < kO3; ++a)
            if (op.out3[a]) bulk_store(op.out3[a] + (row0 + wrow) * 3, s_o3 + a * kRows2 * 3 + wrow * 3, 64 * 3 * sizeof(float));
          bulk_commit();
        }
      } else {
        __syncwarp();
#pragma unroll
        for (int a = 0; a < kO9; ++a)
          if (op.out9[a]) warp_store<9>(op.out9[a] + (row0 + wrow) * 9, s_o9 + a * kRows2 * 9 + wrow * 9, wrows, lane);
#pragma unroll
        for (int a = 0; a < kO3; ++a)
          if (op.out3[a]) warp_store<3>(op.out3[a] + (row0 + wrow) * 3, s_o3 + a * kRows2 * 3 + wrow * 3, wrows, lane);
        __syncwarp();
      }
    }
  }
  bulk_wait_read<0>();
}

template <class Op>
int launch_rowwise_w2(const Op& op, int64_t n, void* stream, const char* name, int ctas_per_sm = 0) {
  if (n < 0) return fail(SO3D_EINVAL, "negative n");
  if (n == 0) return 0;
  int use_tma = 1;
  for (int a = 0; a < Op::kIn9; ++a) {
    if (!op.in9[a]) return fail(SO3D_EINVAL, "null input pointer");
    use_tma &= aligned16(op.in9[a]);
  }
  for (int a = 0; a < Op::kIn3; ++a) {
    if (!op.in3[a]) return fail(SO3D_EINVAL, "null input pointer");
    use_tma &= aligned16(op.in3[a]);
  }
  for (int a = 0; a < Op::kOut9; ++a) use_tma &= aligned16(op.out9[a]);
  for (int a = 0; a < Op::kOut3; ++a) use_tma &= aligned16(op.out3[a]);
  constexpr size_t smem = OpLayout2<Op>::kSmemBytes + (kT2 / 32) * sizeof(uint64_t);  // (+ per-warp barriers of the one-stage mode)
  static_assert(smem <= 227 * 1024, "tile stages exceed shared memory");
  static int resident_dev[kMaxDevices] = {};
  auto kern = rowwise_kernel_w2<Op>;
  const int dev = current_device();
  if (resident_dev[dev] == 0) {
    if (smem > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, kT2, smem) != cudaSuccess || occ < 1) occ = 1;
    resident_dev[dev] = occ;
  }
  if (ctas_per_sm <= 0 || ctas_per_sm > resident_dev[dev]) ctas_per_sm = resident_dev[dev];
  if (const char* e = getenv("SO3D_CTAS_PER_SM")) {
    const int v = atoi(e);
    if (v > 0 && v < ctas_per_sm) ctas_per_sm = v;
  }
  const int64_t tiles = (n + kRows2 - 1) / kRows2;
  const int64_t cap = (int64_t)sm_count() * ctas_per_sm;
  kern<<<(int)(tiles < cap ? tiles : cap), kT2, smem, (cudaStream_t)stream>>>(op, n, use_tma);
  return check_launch(name);
}

// Any one-row op without prefetch hooks on the two-row warp-autonomous engine: the op's row() runs once per row (no packing),
// but the engine work is paid per 64 rows, every warp streams its own slices and there is no CTA barrier in the tile loop.
// Measured at 2^24 rows (profiles/r04r_probe.jsonl, r04s_probe.jsonl; fraction of the HBM peak, one-row -> two-row): ops with
// SMALL outputs gain -- closed-form score 0.85 -> 0.95 (LogpScore2Op, the same construction), log_vec 0.93 -> 0.99, rmat_dist
// 0.97 -> 0.99 -- while ops that write a matrix per row lose, with one or two output stages alike: log_rmat 0.92 -> 0.89,
// exp_vec 0.83 -> 0.79, so3_scale 0.87 -> 0.85, compose 0.98 -> 0.96, shared-row sampler 0.65 -> 0.60 (a warp's 2304-byte
// bulk stores against the CTA-synchronous kernel's 9216-byte ones).  So the choice is per call site (`prefer_two`);
// SO3D_ROW_LANES=1 / 2 forces one kernel for every op (cross-kernel parity test, A/B runs).
#ifndef SO3D_SE3PS_ROWS_TWO
#define SO3D_SE3PS_ROWS_TWO 1  // SE(3) per-row-t reverse step through TwoRow<Op>: 0.731 -> 0.640 ms (r05d); the per-row sampler: 0.232 -> 0.357, stays one-row
#endif
#ifndef SO3D_TWOROW_MINCTAS
#define SO3D_TWOROW_MINCTAS 6
#endif
#ifndef SO3D_TWOROW_OUTSTAGES
#define SO3D_TWOROW_OUTSTAGES 2
#endif
template <class Op>
struct TwoRow : Op {
  struct Pre1 {};
  struct Pre2 {};
  static constexpr int kOutStages = SO3D_TWOROW_OUTSTAGES;
  static constexpr int kInStages = 1;
  static constexpr int kMinCtas = SO3D_TWOROW_MINCTAS;
  int64_t n_rows;  // a row beyond the end must not run (ops read / write per-row scalars by index)
  __device__ Pre1 prefetch1(int64_t) const { return Pre1{}; }
  __device__ Pre2 prefetch2(int64_t, const Pre1&) const { return Pre2{}; }
  __device__ void row2(int64_t i0, const Pre2 (&)[2], const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*o3)[2], const float* tab) const {
    constexpr int kI9 = Op::kIn9, kI3 = Op::kIn3, kO9 = Op::kOut9, kO3 = Op::kOut3;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int64_t i = i0 + 32 * j;
      if (i < n_rows) {
        Mat3 A9[kI9 > 0 ? kI9 : 1], O9[kO9 > 0 ? kO9 : 1];
        Vec3 A3[kI3 > 0 ? kI3 : 1], O3[kO3 > 0 ? kO3 : 1];
#pragma unroll
        for (int a = 0; a < kI9; ++a) A9[a] = a9[a][j];
#pragma unroll
        for (int a = 0; a < kI3; ++a) A3[a] = a3[a][j];
        Op::row(i, A9, A3, O9, O3, tab);
#pragma unroll
        for (int a = 0; a < kO9; ++a) o9[a][j] = O9[a];
#pragma unroll
        for (int a = 0; a < kO3; ++a) o3[a][j] = O3[a];
      }
    }
  }
};
template <class Op>
int launch_rowwise_pick(const Op& op, int64_t n, void* stream, const char* name, bool prefer_two = false) {
  const char* lanes_env = getenv("SO3D_ROW_LANES");  // 1 / 2 force the one-row / two-row kernel for every op
  const int forced = lanes_env ? atoi(lanes_env) : 0;
  if (forced == 1 || (forced != 2 && !prefer_two)) return launch_rowwise(op, n, stream, name);
  TwoRow<Op> op2;
  static_cast<Op&>(op2) = op;
  op2.n_rows = n;
  return launch_rowwise_w2(op2, n, stream, name);
}

#ifndef SO3D_TWOROWPRE_MINCTAS
#define SO3D_TWOROWPRE_MINCTAS 4
#endif
// The same adaptor for one-row ops that DO define prefetch hooks (per-row table rows): the hooks run once per row, row() gets
// the row's Pre2.
template <class Op>
struct TwoRowPre : Op {
  static constexpr int kOutStages = 1;
  static constexpr int kInStages = 1;
  static constexpr int kMinCtas = SO3D_TWOROWPRE_MINCTAS;  // two rows' prefetch state live across the tile: 4 CTAs of 128 threads = 128 registers
  int64_t n_rows;
  __device__ void row2(int64_t i0, const typename Op::Pre2 (&p)[2], const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*o3)[2],
                       const float* tab) const {
    constexpr int kI9 = Op::kIn9, kI3 = Op::kIn3, kO9 = Op::kOut9, kO3 = Op::kOut3;
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int64_t i = i0 + 32 * j;
      if (i < n_rows) {
        Mat3 A9[kI9 > 0 ? kI9 : 1], O9[kO9 > 0 ? kO9 : 1];
        Vec3 A3[kI3 > 0 ? kI3 : 1], O3[kO3 > 0 ? kO3 : 1];
#pragma unroll
        for (int a = 0; a < kI9; ++a) A9[a] = a9[a][j];
#pragma unroll
        for (int a = 0; a < kI3; ++a) A3[a] = a3[a][j];
        Op::row(i, p[j], A9, A3, O9, O3, tab);
#pragma unroll
        for (int a = 0; a < kO9; ++a) o9[a][j] = O9[a];
#pragma unroll
        for (int a = 0; a < kO3; ++a) o3[a][j] = O3[a];
      }
    }
  }
};
template <class Op>
int launch_rowwise_pick_pre(const Op& op, int64_t n, void* stream, const char* name, bool prefer_two) {
  const char* lanes_env = getenv("SO3D_ROW_LANES");
  const int forced = lanes_env ? atoi(lanes_env) : 0;
  if (forced == 1 || (forced != 2 && !prefer_two)) return launch_rowwise(op, n, stream, name);
  TwoRowPre<Op> op2;
  static_cast<Op&>(op2) = op;
  op2.n_rows = n;
  return launch_rowwise_w2(op2, n, stream, name);
}

// dummy arrays for ops without a given kind of operand (zero-length arrays are not allowed)
#define SO3D_OP_ARRAYS(I9, I3, O9, O3) SO3D_OP_ARRAYS_S(I9, I3, O9, O3, 2)
// S = output stages: 2 (double-buffered) or 1 (less shared memory -> more resident CTAs, for latency-bound ops)
#define SO3D_OP_ARRAYS_S(I9, I3, O9, O3, S)                                    \
  static constexpr int kIn9 = I9, kIn3 = I3, kOut9 = O9, kOut3 = O3;           \
  const float* in9[I9 > 0 ? I9 : 1];                                           \
  const float* in3[I3 > 0 ? I3 : 1];                                           \
  float* out9[O9 > 0 ? O9 : 1];                                                \
  float* out3[O3 > 0 ? O3 : 1];                                                \
  static constexpr int kOutStages = S;
// ops without CTA-shared tables
#define SO3D_OP_NO_TAB              \
  static constexpr int kTab = 0;    \
  __device__ void setup(float*) const {}

// ------------------------------------------------------------------------------------------------
// L0 ops
// ------------------------------------------------------------------------------------------------
struct LogOp {  // util.py:164-192
  SO3D_OP_ARRAYS(1, 0, 1, 0)
  SO3D_OP_NO_TAB
  __device__ void row(int64_t, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const { o9[0] = hat(log_vec_fast(a9[0])); }
};
struct LogVecOp {
  SO3D_OP_ARRAYS(1, 0, 0, 1)
  SO3D_OP_NO_TAB
  __device__ void row(int64_t, const Mat3* a9, const Vec3*, Mat3*, Vec3* o3, const float*) const { o3[0] = log_vec_fast(a9[0]); }
};
struct RmatToAaOp {  // util.py:208-219
  SO3D_OP_ARRAYS(1, 0, 0, 1)
  SO3D_OP_NO_TAB
  float* angle;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3*, Vec3* o3, const float*) const {
    const AxisAngleF a = axis_angle_fast(a9[0]);
    o3[0] = a.axis;
    angle[i] = a.theta;
  }
};
struct AaToRmatOp {  // util.py:195-205
  SO3D_OP_ARRAYS(0, 1, 1, 0)
  SO3D_OP_NO_TAB
  const float* angle;
  __device__ void row(int64_t i, const Mat3*, const Vec3* a3, Mat3* o9, Vec3*, const float*) const { o9[0] = aa_to_rmat(a3[0], angle[i]); }
};
struct ExpVecOp {  // diffusion.py:294
  SO3D_OP_ARRAYS(0, 1, 1, 0)
  SO3D_OP_NO_TAB
  __device__ void row(int64_t, const Mat3*, const Vec3* a3, Mat3* o9, Vec3*, const float*) const { o9[0] = quat_to_mat_unit(quat_exp_vec(a3[0])); }
};
struct ScaleOp {  // util.py:349-361
  SO3D_OP_ARRAYS(1, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* s;
  int s_stride;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const { o9[0] = scale_rot_fast(a9[0], s[i * s_stride]); }
};
struct RmatToQuatOp {
  SO3D_OP_ARRAYS(1, 0, 0, 0)
  SO3D_OP_NO_TAB
  float* q;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3*, Vec3*, const float*) const {
    float qq[4];
    rmat_to_quat(a9[0], qq);
    *reinterpret_cast<float4*>(q + 4 * i) = make_float4(qq[0], qq[1], qq[2], qq[3]);
  }
};
struct QuatToRmatOp {  // util.py:222-252
  SO3D_OP_ARRAYS(0, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* q;
  bool q_vec;
  __device__ void row(int64_t i, const Mat3*, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    float4 v;
    if (q_vec) v = __ldcs(reinterpret_cast<const float4*>(q) + i);
    else v = make_float4(q[4 * i], q[4 * i + 1], q[4 * i + 2], q[4 * i + 3]);
    o9[0] = quat_to_rmat(v.x, v.y, v.z, v.w);
  }
};
template <bool TA, bool TB>
__device__ __forceinline__ Mat3 mul_op(const Mat3& a, const Mat3& b) {
  if (TA && TB) {  // A^T B^T = (B A)^T
    const Mat3 c = mul_nn(b, a);
    Mat3 t;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
      for (int j = 0; j < 3; ++j) t.m[3 * i + j] = c.m[3 * j + i];
    return t;
  }
  if (TA) return mul_tn(a, b);
  if (TB) return mul_nt(a, b);
  return mul_nn(a, b);
}
template <bool TA, bool TB>
struct ComposeOp {
  SO3D_OP_ARRAYS(2, 0, 1, 0)
  SO3D_OP_NO_TAB
  __device__ void row(int64_t, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const { o9[0] = mul_op<TA, TB>(a9[0], a9[1]); }
};
// one operand shared by all rows (e.g. mean @ R, distributions.py:50)
template <bool TA, bool TB, bool SharedIsA>
struct ComposeSharedOp {
  SO3D_OP_ARRAYS(1, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* shared;
  __device__ void row(int64_t, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    Mat3 s;
#pragma unroll
    for (int k = 0; k < 9; ++k) s.m[k] = __ldg(shared + k);
    o9[0] = SharedIsA ? mul_op<TA, TB>(s, a9[0]) : mul_op<TA, TB>(a9[0], s);
  }
};
struct RmatDistOp {  // util.py:315-322
  SO3D_OP_ARRAYS(2, 0, 0, 0)
  SO3D_OP_NO_TAB
  float* out;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3*, Vec3*, const float*) const {
    out[i] = 1.41421356237f * axis_angle(mul_tn(a9[0], a9[1])).theta;
  }
};
struct LerpOp {  // util.py:325-338
  SO3D_OP_ARRAYS(2, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* w;
  int w_stride;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    const AxisAngleF a = axis_angle_fast(mul_tn(a9[0], a9[1]));
    o9[0] = mul_nn(a9[0], quat_to_mat_unit(quat_axis_angle(a.axis, w[i * w_stride] * a.theta)));
  }
};

// backward ops
struct LogBwdOp {
  SO3D_OP_ARRAYS(2, 0, 1, 0)
  SO3D_OP_NO_TAB
  __device__ void row(int64_t, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const { o9[0] = log_bwd(a9[0], a9[1]); }
};
struct AaToRmatBwdOp {
  SO3D_OP_ARRAYS(1, 1, 0, 1)
  SO3D_OP_NO_TAB
  const float* angle;
  float* g_angle;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3* a3, Mat3*, Vec3* o3, const float*) const {
    float ga;
    aa_to_rmat_bwd(a3[0], angle[i], a9[0], &o3[0], &ga);
    g_angle[i] = ga;
  }
};
struct ExpVecBwdOp {
  SO3D_OP_ARRAYS(1, 1, 0, 1)
  SO3D_OP_NO_TAB
  __device__ void row(int64_t, const Mat3* a9, const Vec3* a3, Mat3*, Vec3* o3, const float*) const {
    o3[0] = exp_vec_bwd(a3[0], exp_vec(a3[0]), a9[0]);
  }
};
struct ScaleBwdOp {
  // out = exp(hat(s * logvec(R))):  g_s = logvec . Jr^T u,  g_logvec = s Jr^T u, then through the log
  SO3D_OP_ARRAYS(2, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* s;
  int s_stride;
  float* g_s;  // per row (caller reduces for a shared scalar)
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    const float sc = s[i * s_stride];
    const Vec3 lv = log_vec(a9[0]);
    const Vec3 w{sc * lv.x, sc * lv.y, sc * lv.z};
    const Vec3 gw = exp_vec_bwd(w, exp_vec(w), a9[1]);
    if (g_s) g_s[i] = fmaf(lv.x, gw.x, fmaf(lv.y, gw.y, lv.z * gw.z));
    const Vec3 gl{0.5f * sc * gw.x, 0.5f * sc * gw.y, 0.5f * sc * gw.z};  // GL = hat(g_logvec)/2
    o9[0] = log_bwd(a9[0], hat(gl));
  }
};

// ------------------------------------------------------------------------------------------------
// L1: IGSO(3)
// ------------------------------------------------------------------------------------------------
// The HBM-bound evaluators (closed form, auto) request eps one tile ahead through the engine's prefetch hooks: the load
// used to be issued by the row itself and its first use held 32 % of the kernel's stall samples (r03x).  The series
// modes spend microseconds per row and keep their code exactly as it was (ptxas's schedule of the unrolled block is
// sensitive to everything around it, DESIGN.md 4.1).
#ifndef SO3D_LOGP_PREFETCH
#define SO3D_LOGP_PREFETCH 1
#endif
template <bool kOn>
struct LogpPre {};
template <>
struct LogpPre<true> {
  struct Pre1 {};
  struct Pre2 {
    float eps;
  };
};
template <int kMode>
struct LogpScoreOp : LogpPre<SO3D_LOGP_PREFETCH && (kMode == kClosed || kMode == kAuto)> {  // distributions.py:74-77 + score (SURVEY D2), fused with the axis-angle extraction
  SO3D_OP_ARRAYS(1, 0, 0, 1)
  SO3D_OP_NO_TAB
  static constexpr int kMinCtas = (kMode == kClosed || kMode == kAuto) ? 5 : 1;  // HBM-bound evaluators: >= 5 CTAs (<= 51 registers)
#ifndef SO3D_SERIES_WIDE_INDEX
#define SO3D_SERIES_WIDE_INDEX 0  // 1 was 2.6 % faster with the 32-term source form (r01x/r01y); with the 64-term form it is 0.9 % slower
#endif
  static constexpr bool kWideIndex = SO3D_SERIES_WIDE_INDEX && (kMode == kSeries || kMode == kSeriesAdaptive || kMode == kSeriesPure);  // see rowwise_kernel_cta
  const float* eps;
  int eps_stride;
  float* logp;
  float* dlogf;
  int L;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3*, Vec3* o3, const float*) const { row_eps(i, eps[i * eps_stride], a9, o3); }
  __device__ void row_eps(int64_t i, float e, const Mat3* a9, Vec3* o3) const {
    const AxisAngleF a = axis_angle_fast(a9[0]);
    float lf, g;
    igso3_logf_g_t<kMode>(a.theta, e, L, &lf, &g);
    logp[i] = lf;
    if (dlogf) dlogf[i] = g;
    o3[0] = Vec3{g * a.axis.x, g * a.axis.y, g * a.axis.z};
  }
  // prefetch hooks (only instantiated for the modes whose base declares Pre1 / Pre2)
  template <class P1 = typename LogpPre<true>::Pre1>
  __device__ P1 prefetch1(int64_t) const { return P1{}; }
  template <class P1, class P2 = typename LogpPre<true>::Pre2>
  __device__ P2 prefetch2(int64_t i, const P1&) const { return P2{eps[i * eps_stride]}; }
  template <class P2>
  __device__ void row(int64_t i, const P2& p, const Mat3* a9, const Vec3*, Mat3*, Vec3* o3, const float*) const { row_eps(i, p.eps, a9, o3); }
};
// The closed-form / auto evaluators on two rows per thread with per-warp input slices (rowwise_kernel_w2): the engine's
// per-tile work is a third of this light kernel's issue slots and is paid per 64 rows; the axis-angle extraction runs packed
// (axis_angle_fast_l, the same bits), the evaluator itself once per row.  SO3D_LOGP_LANES=1 selects the one-row kernel.
#ifndef SO3D_LOGP2_MINCTAS
#define SO3D_LOGP2_MINCTAS 8
#endif
#ifndef SO3D_LOGP2_AUTO_VOTE
#define SO3D_LOGP2_AUTO_VOTE 1
#endif
#ifndef SO3D_LOGP2_OUTSTAGES
#define SO3D_LOGP2_OUTSTAGES 1
#endif
// The series modes use the same op: both rows' L-term recurrences run as one packed loop (igso3_series_branch_l2, the same
// bits as the one-row kernel).
#ifndef SO3D_SERIES2_MINCTAS
#define SO3D_SERIES2_MINCTAS 4  // register budget of the two-row series kernel (4 CTAs of 128 threads: <= 128 registers)
#endif
template <int kMode>
struct LogpScore2Op : LogpScoreOp<kMode> {
  static constexpr bool kSeriesMode = kMode == kSeries || kMode == kSeriesAdaptive || kMode == kSeriesPure;
  using Pre1 = typename LogpPre<true>::Pre1;
  using Pre2 = typename LogpPre<true>::Pre2;
  static constexpr int kOutStages = SO3D_LOGP2_OUTSTAGES;
  static constexpr int kInStages = 1;
  static constexpr int kMinCtas = kSeriesMode ? SO3D_SERIES2_MINCTAS : SO3D_LOGP2_MINCTAS;
  int64_t n;  // rows beyond the end of a ragged tile must not touch logp / dlogf
  __device__ void row2(int64_t i0, const Pre2 (&p)[2], const Mat3 (*a9)[2], const Vec3 (*)[2], Mat3 (*)[2], Vec3 (*o3)[2], const float*) const {
    const AxisAngleL<L2> a = axis_angle_fast_l(lanes_of(a9[0][0], a9[0][1]));
    float lf2[2], g2[2];
    if constexpr (kSeriesMode) {
      igso3_series_branch_l2<kMode>(a.theta, L2{p[0].eps, p[1].eps}, this->L, lf2, g2);
    } else if (kMode == kAuto && SO3D_LOGP2_AUTO_VOTE) {
      // auto: the closed form for both rows, straight-line; the rows above eps = 1 (none in a DDPM schedule) are re-evaluated by
      // the series behind ONE warp vote instead of a divergent region per row (r05j: the per-row branch scaffolding was 10 % of
      // this kernel's issue slots).  Same bits as igso3_logf_g_t<kAuto>.
      igso3_closed_f32(a.theta.x, p[0].eps, &lf2[0], &g2[0]);
      igso3_closed_f32(a.theta.y, p[1].eps, &lf2[1], &g2[1]);
      const bool s0 = !(p[0].eps <= kAutoSeriesEps), s1 = !(p[1].eps <= kAutoSeriesEps);
      if (__any_sync(__activemask(), s0 || s1)) {
        if (s0) igso3_series_branch<kAuto>(a.theta.x, p[0].eps, this->L, &lf2[0], &g2[0]);
        if (s1) igso3_series_branch<kAuto>(a.theta.y, p[1].eps, this->L, &lf2[1], &g2[1]);
      }
    } else {
      igso3_logf_g_t<kMode>(a.theta.x, p[0].eps, this->L, &lf2[0], &g2[0]);
      igso3_logf_g_t<kMode>(a.theta.y, p[1].eps, this->L, &lf2[1], &g2[1]);
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int64_t i = i0 + 32 * j;
      const float lf = lf2[j], g = g2[j];
      if (i < n) {
        this->logp[i] = lf;
        if (this->dlogf) this->dlogf[i] = g;
      }
      o3[0][j] = j ? Vec3{g * a.axis.x.y, g * a.axis.y.y, g * a.axis.z.y} : Vec3{g * a.axis.x.x, g * a.axis.y.x, g * a.axis.z.x};
    }
  }
};
struct LogpBwdOp {  // SURVEY A.5
  SO3D_OP_ARRAYS(1, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* dlogf;
  const float* gout;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    const Mat3& r = a9[0];
    const float vx = r.m[7] - r.m[5], vy = r.m[2] - r.m[6], vz = r.m[3] - r.m[1];
    const float s = 0.5f * sqrtf(fmaf(vx, vx, fmaf(vy, vy, vz * vz)));
    const float c = 0.5f * (r.m[0] + r.m[4] + r.m[8] - 1.0f);
    const float gg = gout[i] * dlogf[i] / fmaf(s, s, c * c);
    // d theta / dR = [ c/(4 s) (R - R^T) - (s/2) I ] / (s^2 + c^2); at s -> 0 the skew part -> 0/0 * 0
    const float ka = s > 0.f ? gg * c / (4.0f * s) : 0.f;
    const float kd = -0.5f * gg * s;
#pragma unroll
    for (int p = 0; p < 3; ++p)
#pragma unroll
      for (int q = 0; q < 3; ++q) o9[0].m[3 * p + q] = ka * (r.m[3 * p + q] - r.m[3 * q + p]) + (p == q ? kd : 0.f);
  }
};

__global__ void __launch_bounds__(256) density_kernel(const float* __restrict__ omega, const float* __restrict__ eps, int eps_stride,
                                                      float* __restrict__ f, int64_t n, int mode, int L) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    float lf, g;
    igso3_logf_g(omega[i], eps[i * eps_stride], mode, L, &lf, &g);
    f[i] = expf(lf);
  }
}

// Small batches of the series evaluator: ONE WARP per rotation, the L terms split over the 32 lanes (so3d_math.cuh,
// igso3_series_lane): a 4096-row call is 4096 independent 64-term chains instead of 128 warps running 2000-term chains.
template <int kMode>
__global__ void __launch_bounds__(256) series_warp_kernel(const float* __restrict__ R, const float* __restrict__ eps, int eps_stride,
                                                          float* __restrict__ logp, float* __restrict__ score3, float* __restrict__ dlogf,
                                                          int64_t n, int L) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += warps) {
    Mat3 m;
#pragma unroll
    for (int k = 0; k < 9; ++k) m.m[k] = __ldg(R + row * 9 + k);  // same address in every lane: one broadcast transaction each
    const AxisAngleF a = axis_angle_fast(m);
    const float e = __ldg(eps + row * eps_stride);
    float kap, kapp, cexp;
    igso3_series_lane_setup(a.theta, e, &kap, &kapp, &cexp);
    const int Lw = igso3_series_warp_terms(e, L);  // weights beyond it are exactly 0: same bits as all L terms
    SeriesLaneState st = igso3_series_lane(kap, kapp, cexp, lane, igso3_series_lane_terms(Lw), Lw);
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
      st.b += __shfl_xor_sync(0xffffffffu, st.b, off);
      st.d += __shfl_xor_sync(0xffffffffu, st.d, off);
      st.bp += __shfl_xor_sync(0xffffffffu, st.bp, off);
      st.dp += __shfl_xor_sync(0xffffffffu, st.dp, off);
    }
    if (lane == 0) {
      const float F = 2.0f * st.b - st.d, dF = 2.0f * st.bp - st.dp;
      float lf = logf(2.0f * F), g = dF / F;
      if ((kMode == kSeries || kMode == kSeriesAdaptive) && e <= kAutoSeriesEps && a.theta > kSeriesGuard * e) igso3_closed_f32(a.theta, e, &lf, &g);
      logp[row] = lf;
      if (dlogf) dlogf[row] = g;
      if (score3) {
        score3[row * 3] = g * a.axis.x;
        score3[row * 3 + 1] = g * a.axis.y;
        score3[row * 3 + 2] = g * a.axis.z;
      }
    }
  }
}

// distributions.py:15-30.  One CTA per eps row: fp64 density at the 1000 grid points -> fp32, times
// the Haar weight (fp32), trapezoid increments (fp32), prefix sum accumulated in double and rounded
// to float per entry (what ATen's CPU cumsum does for float), normalised by the last entry.
__global__ void __launch_bounds__(256) cdf_table_kernel(const float* __restrict__ eps, const float* __restrict__ grid_loc,
                                                        const float* __restrict__ haar_w, float* __restrict__ trap_out, int quirks) {
  __shared__ float s_pdf[kGrid];
  __shared__ float s_inc[kCdf];
  __shared__ double s_part[8];
  const int row = blockIdx.x;
  const double e = (double)eps[row];
  for (int k = threadIdx.x; k < kGrid; k += blockDim.x) {
    const float loc = grid_loc[k];
    const float dens = (float)igso3_closed_f64((double)loc, e, quirks);  // :19-21 (.float() at :72)
    s_pdf[k] = (loc == 0.0f) ? 0.0f : dens * haar_w[k];                 // :21, :23
  }
  __syncthreads();
  for (int k = threadIdx.x; k < kCdf; k += blockDim.x)
    s_inc[k] = (grid_loc[k + 1] - grid_loc[k]) * (s_pdf[k] + s_pdf[k + 1]) / 2.0f;  // :26-28
  __syncthreads();
  // 8 warps x 125 entries: serial double prefix inside a chunk (lane 0 of each warp), then offsets.
  // Summation order differs from a strictly serial loop only in double precision (error ~1e-16).
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int kChunk = (kCdf + 7) / 8;
  __shared__ double s_pre[kCdf];
  if (lane == 0) {
    double acc = 0.0;
    const int lo = warp * kChunk, hi = min(kCdf, lo + kChunk);
    for (int k = lo; k < hi; ++k) {
      acc += (double)s_inc[k];
      s_pre[k] = acc;
    }
    s_part[warp] = acc;
  }
  __syncthreads();
  double total = 0.0;
  for (int w = 0; w < 8; ++w) total += s_part[w];
  const float last = (float)total;
  for (int k = threadIdx.x; k < kCdf; k += blockDim.x) {
    double off = 0.0;
    const int w = k / kChunk;
    for (int j = 0; j < w; ++j) off += s_part[j];
    const float c = (float)(off + s_pre[k]);
    trap_out[(int64_t)row * kCdf + k] = c / last;  // :29
  }
}

// ------------------------------------------------------------------------------------------------
// CDF tables in shared memory (shared-row fast paths) and the guide builder
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float table_row_angle(const float* __restrict__ cdf, const uint32_t* __restrict__ guide, int64_t row,
                                                 const float* tab, float u) {
  if (guide) {
    const uint4 w = __ldg(reinterpret_cast<const uint4*>(guide) + row * kGuideRecs + guide_bucket(u));  // one 16-byte record
    const GuideRec rec{w.x, __uint_as_float(w.y), __uint_as_float(w.z), __uint_as_float(w.w)};
    return igso3_angle_from_record(cdf + row * kCdf, tab + kTabLoc, rec, u);
  }
  return igso3_angle_from_uniform(cdf + row * kCdf, tab + kTabLoc, u);
}

// distributions.py:15-30 companion: the kGuideRecs guide records of every CDF row (so3d_math.cuh).
__global__ void __launch_bounds__(kTile) cdf_guide_kernel(const float* __restrict__ cdf, uint32_t* __restrict__ guide) {
  __shared__ float s_trap[kGrid];
  const int64_t row = blockIdx.x;
  for (int k = threadIdx.x; k < kCdf; k += kTile) s_trap[k] = cdf[row * kCdf + k];
  __syncthreads();
  uint4* out = reinterpret_cast<uint4*>(guide) + row * kGuideRecs;
  for (int k = threadIdx.x; k < kGuideRecs; k += kTile) {
    const GuideRec r = make_guide_rec(s_trap, k);
    out[k] = make_uint4(r.lohi, __float_as_uint(r.tm1), __float_as_uint(r.t0), __float_as_uint(r.tp1));
  }
}

// ------------------------------------------------------------------------------------------------
// L1: sampling (distributions.py:33-51).  kShared: every sample uses one CDF row (scalar eps).
// ------------------------------------------------------------------------------------------------
// The two halves of SampleOp::row around the angle, for the exact sampler.  (SampleOp keeps its own inline copy: routed
// through these helpers it compiles to different SASS.)
// Axis and uniform of row i: explicit draws where given, else Philox(key, row_offset + i).
__device__ __forceinline__ NoiseDraw sample_draw(const float* u_in, const float* axes_in, const PhiloxKey& key, uint64_t row_offset,
                                                 int64_t i) {
  NoiseDraw out;
  if (axes_in) {
    const float ax = axes_in[3 * i], ay = axes_in[3 * i + 1], az = axes_in[3 * i + 2];
    const float inv = 1.0f / sqrtf(fmaf(ax, ax, fmaf(ay, ay, az * az)));  // distributions.py:36
    out.axis = Vec3{ax * inv, ay * inv, az * inv};
  }
  if (!axes_in || !u_in) {
    const NoiseDraw d = draw_axis_u(key, row_offset + (uint64_t)i);
    if (!axes_in) out.axis = d.axis;
    out.u = d.u;
  }
  if (u_in) out.u = u_in[i];
  return out;
}
// mean @ exp(ang hat(axis)) (distributions.py:38-50) and the optional axis / angle outputs of row i.
__device__ __forceinline__ void sample_finish(Vec3 axis, float ang, const float* mean, int mean_stride, float* angle_out, int64_t i,
                                              Mat3* o9, Vec3* o3) {
  Mat3 out = quat_to_mat_unit(quat_axis_angle(axis, ang));
  if (mean) {
    Mat3 m;
    const float* mp = mean + (mean_stride ? 9 * i : 0);
#pragma unroll
    for (int k = 0; k < 9; ++k) m.m[k] = __ldg(mp + k);
    out = mul_nn(m, out);
  }
  o9[0] = out;
  o3[0] = axis;
  if (angle_out) angle_out[i] = ang;
}

template <bool kShared>
struct SampleOp {
  SO3D_OP_ARRAYS(0, 0, 1, 1)
  static constexpr int kTab = kTabCdfFloats;
  static constexpr bool kWarpSchedule = !kShared;
  const float* cdf;
  const uint32_t* guide;
  const float* loc;
  const int64_t* row_idx;
  int64_t shared_row, rows;
  const float* u_in;
  const float* axes_in;
  PhiloxKey key, key_shift;  // (seed, rng_offset) and its translation stream (rng_offset | 2^63), built by the launcher
  uint64_t row_offset;
  const float* mean;
  int mean_stride;
  float* angle_out;
  __device__ void setup(float* tab) const { stage_cdf(tab, kShared ? cdf + shared_row * kCdf : nullptr, loc); }
  __device__ void row(int64_t i, const Mat3*, const Vec3*, Mat3* o9, Vec3* o3, const float* tab) const {
    Vec3 axis;
    float u;
    if (axes_in) {
      const float ax = axes_in[3 * i], ay = axes_in[3 * i + 1], az = axes_in[3 * i + 2];
      const float inv = 1.0f / sqrtf(fmaf(ax, ax, fmaf(ay, ay, az * az)));  // distributions.py:36
      axis = Vec3{ax * inv, ay * inv, az * inv};
    }
    if (!axes_in || !u_in) {
      const NoiseDraw d = draw_axis_u(key, row_offset + (uint64_t)i);
      if (!axes_in) axis = d.axis;
      u = d.u;
    }
    if (u_in) u = u_in[i];
    float ang;
    if (kShared) {
      ang = shared_row_angle(tab, u);
    } else {
      int64_t rr = row_idx[i];
      rr = rr < 0 ? 0 : (rr >= rows ? rows - 1 : rr);
      ang = table_row_angle(cdf, guide, rr, tab, u);
    }
    Mat3 out = quat_to_mat_unit(quat_axis_angle(axis, ang));
    if (mean) {
      Mat3 m;
      const float* mp = mean + (mean_stride ? 9 * i : 0);
#pragma unroll
      for (int k = 0; k < 9; ++k) m.m[k] = __ldg(mp + k);
      out = mul_nn(m, out);
    }
    o9[0] = out;
    o3[0] = axis;
    if (angle_out) angle_out[i] = ang;
  }
};

// distributions.py:33-51 with the angle from the exact inverse CDF of the IGSO(3) angle law instead of the table
// (igso3_angle_icdf, so3d_math.cuh): per-row or shared eps, nothing staged.  Compute-bound (up to 16 Newton steps of a
// 16-node quadrature or a <= 24-term series per row), so rows run on the warp-autonomous schedule: the step count varies
// per row, and a warp that finishes early streams its outputs without waiting for the CTA.
struct SampleExactOp {
  SO3D_OP_ARRAYS(0, 0, 1, 1)
  SO3D_OP_NO_TAB
  static constexpr bool kWarpSchedule = true;
  const float* eps;
  int eps_stride;
  const float* u_in;
  const float* axes_in;
  PhiloxKey key;  // (seed, rng_offset), built by the launcher: the table sampler's counter layout
  uint64_t row_offset;
  const float* mean;
  int mean_stride;
  float* angle_out;
  __device__ void row(int64_t i, const Mat3*, const Vec3*, Mat3* o9, Vec3* o3, const float*) const {
    const NoiseDraw d = sample_draw(u_in, axes_in, key, row_offset, i);
    sample_finish(d.axis, igso3_angle_icdf(d.u, __ldg(eps + (eps_stride ? i : 0))), mean, mean_stride, angle_out, i, o9, o3);
  }
};

// Backward of the reparameterised exact draw R = mean N, N = exp(w hat(a)), w = F^{-1}(u; eps) at fixed (u, a)
// (IsotropicGaussianSO3.rsample): N is rebuilt from the sampler's axis and angle exactly as SampleExactOp forms it, then
//   G_N = mean^T G,   g_w = <G_N, hat(a) N> = dL/dw,   g_eps = g_w dw/deps (igso3_angle_deps, so3d_math.cuh),   g_mean = G N^T.
// dw/deps is one evaluation of the angle score at the known w, no iteration.  At eps = 0 the angle is 0 for every u and the
// derivative is the eps -> 0+ limit 2 x0(u), so those rows (only those) re-derive u: the given u, else the sampler's Philox
// draw at the same (seed, rng_offset, row_offset).  The per-row cost varies with eps (closed form, series above eps = 1,
// the inversion at eps = 0), so rows run on the warp-autonomous schedule like the sampler.
struct RsampleBwdOp {
  SO3D_OP_ARRAYS(1, 1, 1, 0)
  SO3D_OP_NO_TAB
  static constexpr bool kWarpSchedule = true;
  const float* eps;
  int eps_stride;
  const float* angle;
  const float* mean;
  int mean_stride;
  const float* u_in;
  PhiloxKey key;
  uint64_t row_offset;
  float* g_eps;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3*, const float*) const {
    const float e = __ldg(eps + (eps_stride ? i : 0));
    const float w = __ldg(angle + i);
    const Mat3 nrot = quat_to_mat_unit(quat_axis_angle(a3[0], w));
    Mat3 gn = a9[0];
    if (mean) {
      Mat3 m;
      const float* mp = mean + (mean_stride ? 9 * i : 0);
#pragma unroll
      for (int k = 0; k < 9; ++k) m.m[k] = __ldg(mp + k);
      gn = mul_tn(m, gn);
    }
    const Mat3 dn = mul_nn(hat(a3[0]), nrot);
    float gw = 0.0f;
#pragma unroll
    for (int k = 0; k < 9; ++k) gw = fmaf(gn.m[k], dn.m[k], gw);
    float d;
    if (e == 0.0f) d = igso3_angle_deps_eps0(u_in ? __ldg(u_in + i) : draw_axis_u(key, row_offset + (uint64_t)i).u);
    else d = igso3_angle_deps(w, e);
    g_eps[i] = gw * d;
    o9[0] = mul_nt(a9[0], nrot);
  }
};

// distributions.py:113-127 Bingham.rsample: unit quaternion = normalise(L z), z ~ N(0, I4), L = scale_tril of the
// covariance; fused with util.py:222-252 quat_to_rmat (bingham_train.py:88-90 feeds the samples straight into it).
struct BinghamOp {
  SO3D_OP_ARRAYS(0, 0, 1, 0)
  SO3D_OP_NO_TAB
  const float* tril;  // 4x4 row-major, lower triangle used
  const float* z_in;  // optional explicit normals (n x 4)
  bool z_vec;
  float* q_out;       // optional (n x 4, 16-byte aligned)
  PhiloxKey key, key_shift;  // (seed, rng_offset) and its translation stream (rng_offset | 2^63), built by the launcher
  uint64_t row_offset;
  __device__ void row(int64_t i, const Mat3*, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    Normal4 z;
    if (z_in) {
      const float4 v = z_vec ? __ldcs(reinterpret_cast<const float4*>(z_in) + i)
                             : make_float4(z_in[4 * i], z_in[4 * i + 1], z_in[4 * i + 2], z_in[4 * i + 3]);
      z = Normal4{v.x, v.y, v.z, v.w};
    } else {
      z = normal4_from_u4(philox4x32_10(key, row_offset + (uint64_t)i));
    }
    const float v0 = __ldg(tril + 0) * z.a;
    const float v1 = fmaf(__ldg(tril + 4), z.a, __ldg(tril + 5) * z.b);
    const float v2 = fmaf(__ldg(tril + 8), z.a, fmaf(__ldg(tril + 9), z.b, __ldg(tril + 10) * z.c));
    const float v3 = fmaf(__ldg(tril + 12), z.a, fmaf(__ldg(tril + 13), z.b, fmaf(__ldg(tril + 14), z.c, __ldg(tril + 15) * z.d)));
    const float inv = rsqrt_f(fmaf(v0, v0, fmaf(v1, v1, fmaf(v2, v2, v3 * v3))));  // distributions.py:125
    const float qw = v0 * inv, qx = v1 * inv, qy = v2 * inv, qz = v3 * inv;
    if (q_out) __stcs(reinterpret_cast<float4*>(q_out) + i, make_float4(qw, qx, qy, qz));
    o9[0] = quat_to_rmat(qw, qx, qy, qz);
  }
};

// ------------------------------------------------------------------------------------------------
// L2: fused forward noising (diffusion.py:339-355) and reverse step (diffusion.py:291-326)
// ------------------------------------------------------------------------------------------------
// eps = sqrt_1m_ac[t], noise ~ IGSO3(eps) from cdf row t, x_t = so3_scale(x0, sqrt_ac[t]) @ noise,
// target = vee(log noise)/eps = angle axis / eps (the noise is built from (axis, angle), so its log is known).
// kExtra: the optional noise / score outputs are compiled in (more shared memory per stage).  kDevSeed: the Philox seed
// is read from device memory when the kernel runs (so3d_q_sample_dseed_f32: a captured training step draws fresh noise
// on every replay); a separate instantiation, the by-value kernel's code is untouched.
// kNoiseOut = false with kExtra: the score output without the noise-matrix output (north_star's fused score + noising): no
// second 9-word output stage and no live noise matrix in registers.
template <bool kExtra, bool kDevSeed = false, bool kNoiseOut = kExtra>
struct QSampleOp {
  // per-row table rows are dependent L2 accesses: latency-bound, so favour resident CTAs over output double-buffering
  SO3D_OP_ARRAYS_S(1, 0, (kNoiseOut ? 2 : 1), (kExtra ? 2 : 1), SO3D_QS_OUTSTAGES)  // in: x0;  out9: x_t[, noise];  out3: target[, score]
  static constexpr int kTab = kGrid;  // loc only
  static constexpr int kMinCtas = kExtra ? SO3D_QSX_MINCTAS : SO3D_QS_MINCTAS;  // 4 CTAs (<= 64 registers, no spills) beat 5 CTAs with 56 B of spills: 0.442 vs 0.476 ms (r01m)
  static constexpr bool kWarpSchedule = true;
  const int64_t* t;
  const float* sqrt_ac;
  const float* sqrt_1m_ac;
  int64_t T;
  const float* cdf;
  const uint32_t* guide;
  const float* loc;
  PhiloxKey key, key_shift;  // (seed, rng_offset) and its translation stream (rng_offset | 2^63), built by the launcher
  uint64_t row_offset;
  const uint64_t* seed_dev;  // kDevSeed only
  uint64_t rng_offset;       // kDevSeed only
  __device__ void setup(float* tab) const { stage_cdf(tab, nullptr, loc); }
  // software pipeline: t two tiles ahead; the draw (a pure function of the global row index), the schedule
  // scalars and the guide record one tile ahead -- the row itself then touches no dependent global memory
  // except in the rare multi-point bucket.
  struct Pre1 {
    int64_t t;
  };
  struct Pre2 {
    int ti;
    float eps, sc;
    NoiseDraw d;
    uint4 rec;
  };
  __device__ Pre1 prefetch1(int64_t i) const { return Pre1{t[i]}; }
  __device__ Pre2 prefetch2(int64_t i, const Pre1& p1) const {
    Pre2 p;
    const int64_t ti = p1.t < 0 ? 0 : (p1.t >= T ? T - 1 : p1.t);
    p.ti = (int)ti;
    p.eps = __ldg(sqrt_1m_ac + ti);
    p.sc = __ldg(sqrt_ac + ti);
    if (kDevSeed)
      p.d = draw_axis_u((uint64_t)__ldg(reinterpret_cast<const unsigned long long*>(seed_dev)), row_offset + (uint64_t)i, rng_offset);
    else
      p.d = draw_axis_u(key, row_offset + (uint64_t)i);
    p.rec = guide ? __ldg(reinterpret_cast<const uint4*>(guide) + ti * kGuideRecs + guide_bucket(p.d.u)) : make_uint4(0, 0, 0, 0);
    return p;
  }
  __device__ void row(int64_t, const Pre2& p, const Mat3* a9, const Vec3*, Mat3* o9, Vec3* o3, const float* tab) const {
    const float eps = p.eps;
    const NoiseDraw d = p.d;
    float ang;
    if (guide) {
      const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
      ang = igso3_angle_from_record(cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, d.u);
    } else {
      ang = igso3_angle_from_uniform(cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, d.u);
    }
    const Quat qn = quat_axis_angle(d.axis, ang);
    const AxisAngleF ax = axis_angle_fast(a9[0]);
    o9[0] = quat_to_mat_unit(qmul(quat_axis_angle(ax.axis, p.sc * ax.theta), qn));  // diffusion.py:344-346
    if (kNoiseOut && out9[kNoiseOut ? 1 : 0]) o9[kNoiseOut ? 1 : 0] = quat_to_mat_unit(qn);
    const float k = ang * rcp_approx(eps);                                          // diffusion.py:355
    o3[0] = Vec3{k * d.axis.x, k * d.axis.y, k * d.axis.z};
    if (kExtra && out3[kExtra ? 1 : 0]) {
      float lf, g;
      igso3_logf_g_t<kAuto>(ang, eps, 2000, &lf, &g);
      o3[kExtra ? 1 : 0] = Vec3{g * d.axis.x, g * d.axis.y, g * d.axis.z};
    }
  }
};

// Forward noising on two rows per thread, WARP-AUTONOMOUS (rowwise_kernel_w2): the members, table staging and prefetch
// hooks of QSampleOp (called once per row) and its row arithmetic through the two-lane instantiation of so3d_lanes.cuh
// (q_sample_quat_l: the same IEEE operations per row, hence the same bits as the one-row kernel;
// test_lanes_header_restates_the_scalar_arithmetic_bit_for_bit on the host, test_two_row_noising_equals_one_row on the GPU).
#ifndef SO3D_QS_LANES_DEFAULT2
#define SO3D_QS_LANES_DEFAULT2 1  // forward noising: two rows per thread by default
#endif
#ifndef SO3D_QS2_MINCTAS
#define SO3D_QS2_MINCTAS 4   // 4 CTAs of 128 threads: <= 128 registers
#endif
#ifndef SO3D_QSX2_MINCTAS
#define SO3D_QSX2_MINCTAS 4
#endif
#ifndef SO3D_QS2_ANGLE_VOTE
#define SO3D_QS2_ANGLE_VOTE 1
#endif
#ifndef SO3D_QSX2_AUTO_VOTE
#define SO3D_QSX2_AUTO_VOTE 1
#endif
#ifndef SO3D_QS2_INSTAGES
#define SO3D_QS2_INSTAGES 1  // 1: every warp loads its own slice (rowwise_kernel_w2, kWarpIn): 0.3215 -> 0.3042 ms, with the score 0.386 -> 0.365 (r04j)
#endif
template <bool kExtra, bool kDevSeed = false, bool kNoiseOut = kExtra>
struct QSample2Op : QSampleOp<kExtra, kDevSeed, kNoiseOut> {
  using Base = QSampleOp<kExtra, kDevSeed, kNoiseOut>;
  using Pre2 = typename Base::Pre2;
  static constexpr int kMinCtas = kExtra ? SO3D_QSX2_MINCTAS : SO3D_QS2_MINCTAS;
  static constexpr bool kBranchless = kExtra;  // see OpBranchless
  static constexpr int kInStages = SO3D_QS2_INSTAGES;
  __device__ float angle_of(const Pre2& p, const float* tab) const {
    if (this->guide) {
      const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
      return igso3_angle_from_record(this->cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, p.d.u);
    }
    return igso3_angle_from_uniform(this->cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, p.d.u);
  }
  // both rows' lookups: the one-record resolution straight-line, the rare search (0.2 % of the rows) behind ONE warp vote
  __device__ L2 angles_of(const Pre2 (&p)[2], const float* tab) const {
    // (per variant, r05m: with the score 0.3588 -> 0.3555 ms; plain noising picks a 127-register schedule, 0.304 -> 0.317 ms)
#if SO3D_QS2_ANGLE_VOTE
    if (kExtra && this->guide) {
      const GuideRec r0{p[0].rec.x, __uint_as_float(p[0].rec.y), __uint_as_float(p[0].rec.z), __uint_as_float(p[0].rec.w)};
      const GuideRec r1{p[1].rec.x, __uint_as_float(p[1].rec.y), __uint_as_float(p[1].rec.z), __uint_as_float(p[1].rec.w)};
      bool f0, f1;
      L2 ang{igso3_angle_record_fast(tab + kTabLoc, r0, p[0].d.u, &f0), igso3_angle_record_fast(tab + kTabLoc, r1, p[1].d.u, &f1)};
      if (__any_sync(__activemask(), !f0 || !f1)) {
        if (!f0) ang.x = angle_of(p[0], tab);
        if (!f1) ang.y = angle_of(p[1], tab);
      }
      return ang;
    }
#endif
    return L2{angle_of(p[0], tab), angle_of(p[1], tab)};
  }
  __device__ void row2(int64_t, const Pre2 (&p)[2], const Mat3 (*a9)[2], const Vec3 (*)[2], Mat3 (*o9)[2], Vec3 (*o3)[2], const float* tab) const {
    const L2 ang = angles_of(p, tab);
    const Vec3L<L2> axis{L2{p[0].d.axis.x, p[1].d.axis.x}, L2{p[0].d.axis.y, p[1].d.axis.y}, L2{p[0].d.axis.z, p[1].d.axis.z}};
    QuatL<L2> qn;
    const QuatL<L2> q = q_sample_quat_l<L2>(lanes_of(a9[0][0], a9[0][1]), L2{p[0].sc, p[1].sc}, axis, ang, &qn);  // diffusion.py:344-346
    const Mat3L<L2> o = quat_to_mat_unit_l(q);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      o9[0][0].m[k] = o.m[k].x;
      o9[0][1].m[k] = o.m[k].y;
    }
    if (kNoiseOut && this->out9[kNoiseOut ? 1 : 0]) {
      const Mat3L<L2> nm = quat_to_mat_unit_l(qn);
#pragma unroll
      for (int k = 0; k < 9; ++k) {
        o9[kNoiseOut ? 1 : 0][0].m[k] = nm.m[k].x;
        o9[kNoiseOut ? 1 : 0][1].m[k] = nm.m[k].y;
      }
    }
    const L2 kk{ang.x * rcp_approx(p[0].eps), ang.y * rcp_approx(p[1].eps)};  // diffusion.py:355
    const L2 tx = mul(kk, axis.x), ty = mul(kk, axis.y), tz = mul(kk, axis.z);
    o3[0][0] = Vec3{tx.x, ty.x, tz.x};
    o3[0][1] = Vec3{tx.y, ty.y, tz.y};
    if (kExtra && this->out3[kExtra ? 1 : 0]) {
      // auto evaluator as in LogpScore2Op: closed form for both rows, ONE warp vote for the series override (eps > 1 does not
      // occur in a DDPM schedule: eps_t = sqrt(1 - abar_t)); same bits as igso3_logf_g_t<kAuto> per row
      float lf[2], g[2];
#if SO3D_QSX2_AUTO_VOTE
      igso3_closed_f32(ang.x, p[0].eps, &lf[0], &g[0]);
      igso3_closed_f32(ang.y, p[1].eps, &lf[1], &g[1]);
      const bool s0 = !(p[0].eps <= kAutoSeriesEps), s1 = !(p[1].eps <= kAutoSeriesEps);
      if (__any_sync(__activemask(), s0 || s1)) {
        if (s0) igso3_series_branch<kAuto>(ang.x, p[0].eps, 2000, &lf[0], &g[0]);
        if (s1) igso3_series_branch<kAuto>(ang.y, p[1].eps, 2000, &lf[1], &g[1]);
      }
#else
      igso3_logf_g_t<kAuto>(ang.x, p[0].eps, 2000, &lf[0], &g[0]);
      igso3_logf_g_t<kAuto>(ang.y, p[1].eps, 2000, &lf[1], &g[1]);
#endif
#pragma unroll
      for (int j = 0; j < 2; ++j) o3[kExtra ? 1 : 0][j] = Vec3{g[j] * p[j].d.axis.x, g[j] * p[j].d.axis.y, g[j] * p[j].d.axis.z};
    }
  }
};

// (Forward noising was also tried on two rows per thread with the CTA-synchronous two-row kernel, the step indices
// travelling with the tile: bit-identical, but SLOWER than the warp-autonomous one-row kernel above -- 0.432 vs 0.395 ms per
// 2^24 rows, and 0.688 vs 0.486 ms with the score output (profiles/r03l_qsample_lanes_negative.jsonl): this kernel lives
// on hiding its dependent L2 accesses across tiles, which the CTA-synchronous schedule does not do.  Removed again.)
struct QSampleGivenOp {  // diffusion.py:339-346 with noise supplied
  SO3D_OP_ARRAYS(2, 0, 1, 0)
  SO3D_OP_NO_TAB
  const int64_t* t;
  const float* sqrt_ac;
  int64_t T;
  __device__ void row(int64_t i, const Mat3* a9, const Vec3*, Mat3* o9, Vec3*, const float*) const {
    int64_t ti = t[i];
    ti = ti < 0 ? 0 : (ti >= T ? T - 1 : ti);
    o9[0] = mul_nn(scale_rot(a9[0], __ldg(sqrt_ac + ti)), a9[1]);
  }
};

// Reverse step.  kSharedT: the whole batch shares t (the reference's semantics, Q7): the posterior CDF row and
// its guide live in shared memory; otherwise per-row t with table rows (and the optional guide) read through L2.
// kDevSeed: the Philox seed is read from device memory (CUDA-graph replays with fresh noise, so3d_p_sample_dseed_f32);
// a separate instantiation, so the by-value kernels' code is untouched.
// Per-row t: the row's chain t -> four schedule scalars + guide record used to start inside the row; like forward noising
// it now runs through the engine's prefetch hooks (t two tiles ahead; scalars, draw and record one tile ahead).
#ifndef SO3D_PS_PREFETCH
#define SO3D_PS_PREFETCH 1
#endif
template <bool kOn>
struct PStepPre {};
template <>
struct PStepPre<true> {
  struct Pre1 {
    int64_t t;
  };
  struct Pre2 {
    int ti;
    float k_recip, k_recipm1, k_c1, k_c2;
    NoiseDraw d;
    uint4 rec;
  };
};
template <bool kSharedT, bool kX0, bool kDevSeed = false>
struct PStepOp : PStepPre<SO3D_PS_PREFETCH && !kSharedT> {
  SO3D_OP_ARRAYS_S(1, 1, (kX0 ? 2 : 1), 0, (kSharedT ? SO3D_PSS_OUTSTAGES : 1))  // in: x_t, pred;  out9: x_{t-1}[, x0_hat]
  static constexpr int kTab = kSharedT ? kTabCdfFloats : kGrid;
  // per-row t: cap SO3D_PS_MINCTAS (measured there).  Shared t: issue-bound, shared memory
  // limits it to 4 CTAs and the uncapped 63-register allocation is 3 % faster than a 48-register one (r01l).
  static constexpr int kMinCtas = kSharedT ? SO3D_PSS_MINCTAS : SO3D_PS_MINCTAS;
  static constexpr bool kWarpSchedule = !kSharedT;
  const int64_t* t;
  const float* recip;
  const float* recipm1;
  const float* coef1;
  const float* coef2;
  int64_t T;
  const float* post_cdf;
  const uint32_t* post_guide;
  const float* loc;
  uint64_t seed, rng_offset, row_offset;
  const uint64_t* seed_dev;
  __device__ int64_t clamp_t(int64_t ti) const { return ti < 0 ? 0 : (ti >= T ? T - 1 : ti); }
  // shared t: the step's five scalars are staged once per CTA next to the CDF row (broadcast LDS per tile instead of a
  // dependent t -> schedule chain of global loads and 64-bit address math in every tile: -25 issue slots per warp-tile)
  __device__ void setup(float* tab) const {
    if (post_cdf) stage_cdf(tab, kSharedT ? post_cdf + clamp_t(t[0]) * kCdf : nullptr, loc);
    if (kSharedT && threadIdx.x == 0) {
      const int64_t ti = clamp_t(t[0]);
      tab[kTabScal] = __int_as_float((int)ti);
      tab[kTabScal + 1] = recip[ti];
      tab[kTabScal + 2] = recipm1[ti];
      tab[kTabScal + 3] = coef1[ti];
      tab[kTabScal + 4] = coef2[ti];
      if (kDevSeed) {
        const uint64_t sd = *seed_dev;
        tab[kTabScal + 5] = __uint_as_float((uint32_t)sd);
        tab[kTabScal + 6] = __uint_as_float((uint32_t)(sd >> 32));
      }
    }
  }
  __device__ void row(int64_t i, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3*, const float* tab) const {
    int64_t ti;
    float k_recip, k_recipm1, k_c1, k_c2;
    if (kSharedT) {
      ti = __float_as_int(tab[kTabScal]);
      k_recip = tab[kTabScal + 1], k_recipm1 = tab[kTabScal + 2], k_c1 = tab[kTabScal + 3], k_c2 = tab[kTabScal + 4];
    } else {
      ti = clamp_t(t[i]);
      k_recip = __ldg(recip + ti), k_recipm1 = __ldg(recipm1 + ti), k_c1 = __ldg(coef1 + ti), k_c2 = __ldg(coef2 + ti);
    }
    Quat qh;
    Quat qm = p_mean_quat(a9[0], a3[0], k_recip, k_recipm1, k_c1, k_c2, &qh);
    if (post_cdf && ti != 0) {                                                     // diffusion.py:320-326
      // (the launcher-side key schedule the other ops use measured 2 % slower here: ptxas then allocates 46 instead of
      // 63 registers and schedules with less overlap, profiles/r01w_probe_engine.jsonl)
      const uint64_t sd = (kDevSeed && kSharedT)
                              ? ((uint64_t)__float_as_uint(tab[kTabScal + 5]) | ((uint64_t)__float_as_uint(tab[kTabScal + 6]) << 32))
                              : seed;
      const NoiseDraw d = draw_axis_u(sd, row_offset + (uint64_t)i, rng_offset);
      const float ang = kSharedT ? shared_row_angle(tab, d.u) : table_row_angle(post_cdf, post_guide, ti, tab, d.u);
      qm = qmul(qm, quat_axis_angle(d.axis, ang));
    }
    o9[0] = quat_to_mat_unit(qm);
    if (kX0) o9[kX0 ? 1 : 0] = quat_to_mat_unit(qh);
  }
  // prefetch hooks of the per-row-t instantiations (the same functions of the same inputs as row() above: same bits)
  template <class P1 = typename PStepPre<true>::Pre1>
  __device__ P1 prefetch1(int64_t i) const { return P1{t[i]}; }
  template <class P1, class P2 = typename PStepPre<true>::Pre2>
  __device__ P2 prefetch2(int64_t i, const P1& p1) const {
    P2 p;
    const int64_t ti = clamp_t(p1.t);
    p.ti = (int)ti;
    p.k_recip = __ldg(recip + ti), p.k_recipm1 = __ldg(recipm1 + ti), p.k_c1 = __ldg(coef1 + ti), p.k_c2 = __ldg(coef2 + ti);
    p.d = draw_axis_u(seed, row_offset + (uint64_t)i, rng_offset);
    p.rec = (post_cdf && post_guide) ? __ldg(reinterpret_cast<const uint4*>(post_guide) + ti * kGuideRecs + guide_bucket(p.d.u)) : make_uint4(0, 0, 0, 0);
    return p;
  }
  template <class P2>
  __device__ void row(int64_t, const P2& p, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3*, const float* tab) const {
    Quat qh;
    Quat qm = p_mean_quat(a9[0], a3[0], p.k_recip, p.k_recipm1, p.k_c1, p.k_c2, &qh);
    if (post_cdf && p.ti != 0) {  // diffusion.py:320-326
      float ang;
      if (post_guide) {
        const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
        ang = igso3_angle_from_record(post_cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, p.d.u);
      } else {
        ang = igso3_angle_from_uniform(post_cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, p.d.u);
      }
      qm = qmul(qm, quat_axis_angle(p.d.axis, ang));
    }
    o9[0] = quat_to_mat_unit(qm);
    if (kX0) o9[kX0 ? 1 : 0] = quat_to_mat_unit(qh);
  }
};

// The per-row-t reverse step on two rows per thread, warp-autonomous (rowwise_kernel_w2): members and prefetch hooks of
// PStepOp<false, false>, row arithmetic through p_mean_quat_l<L2> (same bits; test_two_row_reverse_step_rows_equals_one_row).
#ifndef SO3D_PS2R_MINCTAS
#define SO3D_PS2R_MINCTAS 4
#endif
#ifndef SO3D_PS2R_INSTAGES
#define SO3D_PS2R_INSTAGES 1  // per-warp input slices: 0.382 -> 0.372 ms (r04j)
#endif
template <bool kDevSeed>
struct PStepRows2Op : PStepOp<false, false, kDevSeed> {
  using Base = PStepOp<false, false, kDevSeed>;
  using Pre2 = typename Base::Pre2;
  static constexpr int kMinCtas = SO3D_PS2R_MINCTAS;
  static constexpr int kInStages = SO3D_PS2R_INSTAGES;
  __device__ float angle_of(const Pre2& p, const float* tab) const {
    if (this->post_guide) {
      const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
      return igso3_angle_from_record(this->post_cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, p.d.u);
    }
    return igso3_angle_from_uniform(this->post_cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, p.d.u);
  }
  __device__ void row2(int64_t, const Pre2 (&p)[2], const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*)[2], const float* tab) const {
    const Mat3L<L2> x = lanes_of(a9[0][0], a9[0][1]);
    const Vec3L<L2> pred{L2{a3[0][0].x, a3[0][1].x}, L2{a3[0][0].y, a3[0][1].y}, L2{a3[0][0].z, a3[0][1].z}};
    QuatL<L2> qh;
    QuatL<L2> qm = p_mean_quat_rows_l(x, pred, L2{p[0].k_recip, p[1].k_recip}, L2{p[0].k_recipm1, p[1].k_recipm1}, L2{p[0].k_c1, p[1].k_c1},
                                      L2{p[0].k_c2, p[1].k_c2}, &qh);
    if (this->post_cdf) {  // diffusion.py:320-326; rows at t == 0 take the mean
      const bool n0 = p[0].ti != 0, n1 = p[1].ti != 0;
      if (n0 || n1) {
        const L2 ang{n0 ? angle_of(p[0], tab) : 0.f, n1 ? angle_of(p[1], tab) : 0.f};
        const Vec3L<L2> axis{L2{p[0].d.axis.x, p[1].d.axis.x}, L2{p[0].d.axis.y, p[1].d.axis.y}, L2{p[0].d.axis.z, p[1].d.axis.z}};
        const QuatL<L2> qz = qmul_l(qm, quat_axis_angle_l(axis, ang));
        qm.w = L2{n0 ? qz.w.x : qm.w.x, n1 ? qz.w.y : qm.w.y};
        qm.x = L2{n0 ? qz.x.x : qm.x.x, n1 ? qz.x.y : qm.x.y};
        qm.y = L2{n0 ? qz.y.x : qm.y.x, n1 ? qz.y.y : qm.y.y};
        qm.z = L2{n0 ? qz.z.x : qm.z.x, n1 ? qz.z.y : qm.z.y};
      }
    }
    const Mat3L<L2> o = quat_to_mat_unit_l(qm);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      o9[0][0].m[k] = o.m[k].x;
      o9[0][1].m[k] = o.m[k].y;
    }
  }
};

// The shared-t reverse step on two rows per thread (rowwise_kernel_cta2): the arithmetic of PStepOp<true, false> through the
// two-lane instantiations of so3d_lanes.cuh -- the same IEEE operations per row, hence the same bits.
// Measured on B200, 2^24 rows (profiles/r03k_pstep_lanes.jsonl): one row per thread 0.3446 ms; two rows per thread with
// 256 threads / 512-row tiles (2 resident CTAs) 0.3478; 128 threads / 256-row tiles, two output stages (4 CTAs) 0.3346; one
// output stage (44 KB of shared memory -> 5 CTAs of 4 warps) 0.3217 ms; and with ONE input stage as well (refilled as soon
// as the rows of the current tile are in registers: 31.6 KB -> 7 CTAs, 28 warps) 0.3094 ms = 5.42e10 particle-steps/s =
// 0.695 of the HBM roofline (profiles/r03o_pstep_instages.jsonl; two output stages on top of that: 0.3241).
#ifndef SO3D_PSS2_OUTSTAGES
#define SO3D_PSS2_OUTSTAGES 1
#endif
#ifndef SO3D_PSS2_MINCTAS
#define SO3D_PSS2_MINCTAS 7
#endif
#ifndef SO3D_PSS2_INSTAGES
#define SO3D_PSS2_INSTAGES 1
#endif
template <bool kDevSeed>
struct PStep2Op {
  SO3D_OP_ARRAYS_S(1, 1, 1, 0, SO3D_PSS2_OUTSTAGES)  // in: x_t, pred;  out9: x_{t-1}
  static constexpr int kTab = kTabCdfFloats;
  static constexpr int kMinCtas = SO3D_PSS2_MINCTAS;
  static constexpr int kInStages = SO3D_PSS2_INSTAGES;
  const int64_t* t;
  const float* recip;
  const float* recipm1;
  const float* coef1;
  const float* coef2;
  int64_t T;
  const float* post_cdf;
  const float* loc;
  uint64_t seed, rng_offset, row_offset;
  const uint64_t* seed_dev;
  __device__ int64_t clamp_t(int64_t ti) const { return ti < 0 ? 0 : (ti >= T ? T - 1 : ti); }
  __device__ void setup(float* tab) const {
    if (post_cdf) stage_cdf(tab, post_cdf + clamp_t(t[0]) * kCdf, loc);
    if (threadIdx.x == 0) {
      const int64_t ti = clamp_t(t[0]);
      tab[kTabScal] = __int_as_float((int)ti);
      tab[kTabScal + 1] = recip[ti];
      tab[kTabScal + 2] = recipm1[ti];
      tab[kTabScal + 3] = coef1[ti];
      tab[kTabScal + 4] = coef2[ti];
      if (kDevSeed) {
        const uint64_t sd = *seed_dev;
        tab[kTabScal + 5] = __uint_as_float((uint32_t)sd);
        tab[kTabScal + 6] = __uint_as_float((uint32_t)(sd >> 32));
      }
    }
  }
  __device__ void row2(int64_t i0, const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*)[2], const float* tab) const {
    row2_at<kT2>(i0, a9, a3, o9, tab);
  }
  template <int kLane1>  // lane 1 is the row i0 + kLane1
  __device__ void row2_at(int64_t i0, const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], const float* tab) const {
    const int ti = __float_as_int(tab[kTabScal]);
    const float k_recip = tab[kTabScal + 1], k_recipm1 = tab[kTabScal + 2], k_c1 = tab[kTabScal + 3], k_c2 = tab[kTabScal + 4];
    const Mat3L<L2> x = lanes_of(a9[0][0], a9[0][1]);
    const Vec3L<L2> pred{L2{a3[0][0].x, a3[0][1].x}, L2{a3[0][0].y, a3[0][1].y}, L2{a3[0][0].z, a3[0][1].z}};
    QuatL<L2> qh;
    QuatL<L2> qm = p_mean_quat_l<L2, true>(x, pred, k_recip, k_recipm1, k_c1, k_c2, &qh);
    if (post_cdf && ti != 0) {  // diffusion.py:320-326
      const uint64_t sd = kDevSeed ? ((uint64_t)__float_as_uint(tab[kTabScal + 5]) | ((uint64_t)__float_as_uint(tab[kTabScal + 6]) << 32)) : seed;
      const uint64_t row = row_offset + (uint64_t)i0;
      const U4 r0 = philox4x32_10(sd, row, rng_offset), r1 = philox4x32_10(sd, row + kLane1, rng_offset);
      const Vec3L<L2> axis = sphere_from_uniforms_l(L2{u01(r0.x), u01(r1.x)}, L2{u01(r0.y), u01(r1.y)});
      const L2 ang{shared_row_angle(tab, u01(r0.z)), shared_row_angle(tab, u01(r1.z))};
      qm = qmul_l(qm, quat_axis_angle_l(axis, ang));
    }
    const Mat3L<L2> o = quat_to_mat_unit_l(qm);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      o9[0][0].m[k] = o.m[k].x;
      o9[0][1].m[k] = o.m[k].y;
    }
  }
};

// Experiment (SO3D_PSTEP_ENGINE=w2): the same step on the warp-autonomous two-row engine -- no CTA barriers, but two input
// stages (44 KB -> 5 CTAs of 4 warps instead of 7).
#ifndef SO3D_PSS2W_INSTAGES
#define SO3D_PSS2W_INSTAGES 1
#endif
template <bool kDevSeed>
struct PStep2wOp : PStep2Op<kDevSeed> {
  struct Pre1 {};
  struct Pre2 {};
  static constexpr int kInStages = SO3D_PSS2W_INSTAGES;
  static constexpr int kMinCtas = SO3D_PSS2W_INSTAGES == 1 ? 7 : 5;
  __device__ Pre1 prefetch1(int64_t) const { return Pre1{}; }
  __device__ Pre2 prefetch2(int64_t, const Pre1&) const { return Pre2{}; }
  __device__ void row2(int64_t i0, const Pre2 (&)[2], const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*)[2], const float* tab) const {
    this->template row2_at<32>(i0, a9, a3, o9, tab);
  }
};

// ------------------------------------------------------------------------------------------------
// SE(3) arm (SURVEY 8f-3): diffusion.py:432-573 SE3Diffusion / distributions.py:84-110 IGSO3xR3.  The rotation
// half is the SO(3) arithmetic above; the translation half is a scalar DDPM in R^3 with noise scale
// eps * shift_scale, carried by the same launch (three more 12-byte arrays per row).
// The translation normals come from a second Philox block of the same row: counter (row, rng_offset | 2^63), so the
// rotation draws are bit-identical to the SO(3)-only kernels at the same (seed, rng_offset).
// ------------------------------------------------------------------------------------------------
constexpr uint64_t kShiftStream = 0x8000000000000000ull;

// kDevSeed of the SE(3) ops: the Philox seed is read from device memory when the kernel runs (so3d_se3_*_dseed_f32: a
// captured training step or sampling loop draws fresh noise on every replay).  Both streams come from it, the rotation
// block at (row, rng_offset) and the translation block at (row, rng_offset | 2^63): the draws of the by-value kernels at
// seed = *seed_dev.  The by-value instantiations derive from the empty DevSeedArgs<false>, so their layout and code are
// those of the plain structs.
template <bool kDevSeed>
struct DevSeedArgs {};
template <>
struct DevSeedArgs<true> {
  const uint64_t* seed_dev;
  uint64_t rng_offset;
  __device__ uint64_t load_seed() const { return (uint64_t)__ldg(reinterpret_cast<const unsigned long long*>(seed_dev)); }
};
// the seed a shared-t reverse step staged next to its scalars (two words after the six of the SE(3) step)
__device__ __forceinline__ uint64_t staged_seed(const float* tab) {
  return (uint64_t)__float_as_uint(tab[kTabScal + 6]) | ((uint64_t)__float_as_uint(tab[kTabScal + 7]) << 32);
}

// q_sample + p_losses targets: diffusion.py:498-516
//   rot_t = so3_scale(rot0, a_t) @ noise_rot;  target_rot = vee(log noise_rot)/eps_t
//   shift_t = a_t shift0 + eps_t shift_scale z;  target_shift = noise_shift/(eps_t shift_scale) = z
template <bool kDevSeed = false>
struct SE3QSampleOp : DevSeedArgs<kDevSeed> {
  SO3D_OP_ARRAYS_S(1, 1, 1, 3, 1)  // in: rot0 | shift0;  out: rot_t | target_rot, shift_t, target_shift
  static constexpr int kTab = kGrid;
  static constexpr bool kWarpSchedule = true;
#ifndef SO3D_SE3QS_MINCTAS
#define SO3D_SE3QS_MINCTAS 3
#endif
  static constexpr int kMinCtas = SO3D_SE3QS_MINCTAS;
  const int64_t* t;
  const float* sqrt_ac;
  const float* sqrt_1m_ac;
  int64_t T;
  const float* cdf;
  const uint32_t* guide;
  const float* loc;
  float shift_scale;
  PhiloxKey key, key_shift;  // (seed, rng_offset) and its translation stream (rng_offset | 2^63), built by the launcher
  uint64_t row_offset;
  __device__ void setup(float* tab) const { stage_cdf(tab, nullptr, loc); }
  // the rotation draw and the translation block of global row r
  __device__ NoiseDraw rot_draw(uint64_t r) const {
    if constexpr (kDevSeed) return draw_axis_u(this->load_seed(), r, this->rng_offset);
    else return draw_axis_u(key, r);
  }
  __device__ U4 shift_block(uint64_t r) const {
    if constexpr (kDevSeed) return philox4x32_10(this->load_seed(), r, this->rng_offset | kShiftStream);
    else return philox4x32_10(key_shift, r);
  }
#ifndef SO3D_SE3QS_PREFETCH
#define SO3D_SE3QS_PREFETCH 1  // the software pipeline of QSampleOp: t two tiles ahead, draw + schedule scalars + guide record one tile ahead
#endif
#if SO3D_SE3QS_PREFETCH
  struct Pre1 {
    int64_t t;
  };
  struct Pre2 {
    int ti;
    float eps, sc;
    NoiseDraw d;
    uint4 rec;
  };
  __device__ Pre1 prefetch1(int64_t i) const { return Pre1{t[i]}; }
  __device__ Pre2 prefetch2(int64_t i, const Pre1& p1) const {
    Pre2 p;
    const int64_t ti = p1.t < 0 ? 0 : (p1.t >= T ? T - 1 : p1.t);
    p.ti = (int)ti;
    p.eps = __ldg(sqrt_1m_ac + ti);
    p.sc = __ldg(sqrt_ac + ti);
    p.d = rot_draw(row_offset + (uint64_t)i);
    p.rec = guide ? __ldg(reinterpret_cast<const uint4*>(guide) + ti * kGuideRecs + guide_bucket(p.d.u)) : make_uint4(0, 0, 0, 0);
    return p;
  }
  __device__ void row(int64_t i, const Pre2& p, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3* o3, const float* tab) const {
    const float eps = p.eps, sc = p.sc;
    const NoiseDraw d = p.d;
    float ang;
    if (guide) {
      const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
      ang = igso3_angle_from_record(cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, d.u);
    } else {
      ang = igso3_angle_from_uniform(cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, d.u);
    }
#else
  __device__ void row(int64_t i, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3* o3, const float* tab) const {
    int64_t ti = t[i];
    ti = ti < 0 ? 0 : (ti >= T ? T - 1 : ti);
    const float eps = __ldg(sqrt_1m_ac + ti), sc = __ldg(sqrt_ac + ti);
    const NoiseDraw d = rot_draw(row_offset + (uint64_t)i);
    const float ang = table_row_angle(cdf, guide, ti, tab, d.u);
#endif
    const Quat qn = quat_axis_angle(d.axis, ang);
    const AxisAngleF ax = axis_angle_fast(a9[0]);
    o9[0] = quat_to_mat_unit(qmul(quat_axis_angle(ax.axis, sc * ax.theta), qn));
    const float k = ang * rcp_approx(eps);
    o3[0] = Vec3{k * d.axis.x, k * d.axis.y, k * d.axis.z};
    const Normal4 z = normal4_from_u4(shift_block(row_offset + (uint64_t)i));
    const float ns = eps * shift_scale;
    o3[1] = Vec3{fmaf(sc, a3[0].x, ns * z.a), fmaf(sc, a3[0].y, ns * z.b), fmaf(sc, a3[0].z, ns * z.c)};
    o3[2] = Vec3{z.a, z.b, z.c};
  }
};

#if SO3D_SE3QS_PREFETCH
// SE(3) noising on two rows per thread, warp-autonomous (rowwise_kernel_w2): same bits as SE3QSampleOp
// (test_two_row_se3_noising_equals_one_row).
#ifndef SO3D_SE3QS2_MINCTAS
#define SO3D_SE3QS2_MINCTAS 3  // 135 registers; the 119-register schedule of a 4-CTA cap is 10 % slower (r04g, r04k)
#endif
#ifndef SO3D_SE3QS2_BRANCHLESS
#define SO3D_SE3QS2_BRANCHLESS 0
#endif
#ifndef SO3D_SE3QS2_INSTAGES
#define SO3D_SE3QS2_INSTAGES 1
#endif
template <bool kDevSeed = false>
struct SE3QSample2Op : SE3QSampleOp<kDevSeed> {
  using Base = SE3QSampleOp<kDevSeed>;
  using Pre2 = typename Base::Pre2;
  static constexpr int kMinCtas = SO3D_SE3QS2_MINCTAS;
  static constexpr int kInStages = SO3D_SE3QS2_INSTAGES;
  static constexpr bool kBranchless = SO3D_SE3QS2_BRANCHLESS;
  __device__ float angle_of(const Pre2& p, const float* tab) const {
    if (this->guide) {
      const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
      return igso3_angle_from_record(this->cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, p.d.u);
    }
    return igso3_angle_from_uniform(this->cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, p.d.u);
  }
  __device__ void row2(int64_t i0, const Pre2 (&p)[2], const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*o3)[2], const float* tab) const {
    const L2 ang{angle_of(p[0], tab), angle_of(p[1], tab)};
    const Vec3L<L2> axis{L2{p[0].d.axis.x, p[1].d.axis.x}, L2{p[0].d.axis.y, p[1].d.axis.y}, L2{p[0].d.axis.z, p[1].d.axis.z}};
    const L2 eps{p[0].eps, p[1].eps}, sc{p[0].sc, p[1].sc};
    QuatL<L2> qn;
    const Mat3L<L2> o = quat_to_mat_unit_l(q_sample_quat_l<L2>(lanes_of(a9[0][0], a9[0][1]), sc, axis, ang, &qn));
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      o9[0][0].m[k] = o.m[k].x;
      o9[0][1].m[k] = o.m[k].y;
    }
    const L2 kk{ang.x * rcp_approx(eps.x), ang.y * rcp_approx(eps.y)};
    const L2 tx = mul(kk, axis.x), ty = mul(kk, axis.y), tz = mul(kk, axis.z);
    o3[0][0] = Vec3{tx.x, ty.x, tz.x};
    o3[0][1] = Vec3{tx.y, ty.y, tz.y};
    const Normal4 z0 = normal4_from_u4(this->shift_block(this->row_offset + (uint64_t)i0));
    const Normal4 z1 = normal4_from_u4(this->shift_block(this->row_offset + (uint64_t)i0 + 32u));
    const L2 ns = mul(eps, bc<L2>(this->shift_scale));
    const L2 sx = fma(sc, L2{a3[0][0].x, a3[0][1].x}, mul(ns, L2{z0.a, z1.a}));
    const L2 sy = fma(sc, L2{a3[0][0].y, a3[0][1].y}, mul(ns, L2{z0.b, z1.b}));
    const L2 sz = fma(sc, L2{a3[0][0].z, a3[0][1].z}, mul(ns, L2{z0.c, z1.c}));
    o3[1][0] = Vec3{sx.x, sy.x, sz.x};
    o3[1][1] = Vec3{sx.y, sy.y, sz.y};
    o3[2][0] = Vec3{z0.a, z0.b, z0.c};
    o3[2][1] = Vec3{z1.a, z1.b, z1.c};
  }
};
#endif

// reverse step: diffusion.py:446-485
//   rot as PStepOp;  shift0_hat = recip_t shift_t - recipm1_t pred_shift;  mean = c1 shift0_hat + c2 shift_t;
//   out = t == 0 ? mean : mean + sigma_t shift_scale z
#ifndef SO3D_SE3PS_PREFETCH
#define SO3D_SE3PS_PREFETCH 1  // per-row t: step index two tiles ahead, schedule scalars + draw + guide record one tile ahead
#endif
template <bool kOn>
struct SE3PStepPre {};
template <>
struct SE3PStepPre<true> {
  struct Pre1 {
    int64_t t;
  };
  struct Pre2 {
    int ti;
    float k_recip, k_recipm1, k_c1, k_c2, k_sigma;
    NoiseDraw d;
    uint4 rec;
  };
};
// kDevSeed (shared t only): the seed is read from seed_dev once per CTA in setup and staged next to the step's scalars.
template <bool kSharedT, bool kDevSeed = false>
struct SE3PStepOp : SE3PStepPre<SO3D_SE3PS_PREFETCH && !kSharedT>, DevSeedArgs<kDevSeed> {
  static_assert(kSharedT || !kDevSeed, "the device-seed reverse step takes a shared step index");
  SO3D_OP_ARRAYS_S(1, 3, 1, 1, 1)  // in: rot_t | pred_rot, shift_t, pred_shift;  out: rot | shift
  static constexpr int kTab = kSharedT ? kTabCdfFloats : kGrid;
  // per-row t: cap SO3D_PS_MINCTAS (measured there).  Shared t: issue-bound, shared memory
  // limits it to 4 CTAs and the uncapped 63-register allocation is 3 % faster than a 48-register one (r01l).
  static constexpr int kMinCtas = kSharedT ? SO3D_PSS_MINCTAS : SO3D_PS_MINCTAS;
  static constexpr bool kWarpSchedule = !kSharedT;
  const int64_t* t;
  const float* recip;
  const float* recipm1;
  const float* coef1;
  const float* coef2;
  const float* sigma;
  int64_t T;
  const float* post_cdf;
  const uint32_t* post_guide;
  const float* loc;
  float shift_scale;
  PhiloxKey key, key_shift;  // (seed, rng_offset) and its translation stream (rng_offset | 2^63), built by the launcher
  uint64_t row_offset;
  __device__ int64_t clamp_t(int64_t ti) const { return ti < 0 ? 0 : (ti >= T ? T - 1 : ti); }
  __device__ void setup(float* tab) const {
    if (post_cdf) stage_cdf(tab, kSharedT ? post_cdf + clamp_t(t[0]) * kCdf : nullptr, loc);
    if (kSharedT && threadIdx.x == 0) {  // the step's scalars, staged once per CTA (see PStepOp)
      const int64_t ti = clamp_t(t[0]);
      tab[kTabScal] = __int_as_float((int)ti);
      tab[kTabScal + 1] = recip[ti];
      tab[kTabScal + 2] = recipm1[ti];
      tab[kTabScal + 3] = coef1[ti];
      tab[kTabScal + 4] = coef2[ti];
      tab[kTabScal + 5] = sigma[ti];
      if constexpr (kDevSeed) {
        const uint64_t sd = *this->seed_dev;
        tab[kTabScal + 6] = __uint_as_float((uint32_t)sd);
        tab[kTabScal + 7] = __uint_as_float((uint32_t)(sd >> 32));
      }
    }
  }
  // the rotation draw and the translation block of global row r (kDevSeed: from the staged seed)
  __device__ NoiseDraw rot_draw(uint64_t r, const float* tab) const {
    if constexpr (kDevSeed) return draw_axis_u(staged_seed(tab), r, this->rng_offset);
    else return draw_axis_u(key, r);
  }
  __device__ U4 shift_block(uint64_t r, const float* tab) const {
    if constexpr (kDevSeed) return philox4x32_10(staged_seed(tab), r, this->rng_offset | kShiftStream);
    else return philox4x32_10(key_shift, r);
  }
  __device__ void row(int64_t i, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3* o3, const float* tab) const {
    int64_t ti;
    float k_recip, k_recipm1, k_c1, k_c2, k_sigma;
    if (kSharedT) {
      ti = __float_as_int(tab[kTabScal]);
      k_recip = tab[kTabScal + 1], k_recipm1 = tab[kTabScal + 2], k_c1 = tab[kTabScal + 3], k_c2 = tab[kTabScal + 4], k_sigma = tab[kTabScal + 5];
    } else {
      ti = clamp_t(t[i]);
      k_recip = __ldg(recip + ti), k_recipm1 = __ldg(recipm1 + ti), k_c1 = __ldg(coef1 + ti), k_c2 = __ldg(coef2 + ti), k_sigma = __ldg(sigma + ti);
    }
    Quat qh;
    Quat qm = p_mean_quat(a9[0], a3[0], k_recip, k_recipm1, k_c1, k_c2, &qh);
    const Vec3 st = a3[1], ps = a3[2];
    Vec3 m;
    m.x = fmaf(k_c1, fmaf(k_recip, st.x, -k_recipm1 * ps.x), k_c2 * st.x);
    m.y = fmaf(k_c1, fmaf(k_recip, st.y, -k_recipm1 * ps.y), k_c2 * st.y);
    m.z = fmaf(k_c1, fmaf(k_recip, st.z, -k_recipm1 * ps.z), k_c2 * st.z);
    if (post_cdf && ti != 0) {
      const NoiseDraw d = rot_draw(row_offset + (uint64_t)i, tab);
      const float ang = kSharedT ? shared_row_angle(tab, d.u) : table_row_angle(post_cdf, post_guide, ti, tab, d.u);
      qm = qmul(qm, quat_axis_angle(d.axis, ang));
      const Normal4 z = normal4_from_u4(shift_block(row_offset + (uint64_t)i, tab));
      const float ns = k_sigma * shift_scale;
      m = Vec3{fmaf(ns, z.a, m.x), fmaf(ns, z.b, m.y), fmaf(ns, z.c, m.z)};
    }
    o9[0] = quat_to_mat_unit(qm);
    o3[0] = m;
  }
  // prefetch hooks of the per-row-t instantiation (same functions of the same inputs as row(): same bits)
  template <class P1 = typename SE3PStepPre<true>::Pre1>
  __device__ P1 prefetch1(int64_t i) const { return P1{t[i]}; }
  template <class P1, class P2 = typename SE3PStepPre<true>::Pre2>
  __device__ P2 prefetch2(int64_t i, const P1& p1) const {
    P2 p;
    const int64_t ti = clamp_t(p1.t);
    p.ti = (int)ti;
    p.k_recip = __ldg(recip + ti), p.k_recipm1 = __ldg(recipm1 + ti), p.k_c1 = __ldg(coef1 + ti), p.k_c2 = __ldg(coef2 + ti), p.k_sigma = __ldg(sigma + ti);
    p.d = draw_axis_u(key, row_offset + (uint64_t)i);
    p.rec = (post_cdf && post_guide) ? __ldg(reinterpret_cast<const uint4*>(post_guide) + ti * kGuideRecs + guide_bucket(p.d.u)) : make_uint4(0, 0, 0, 0);
    return p;
  }
  template <class P2>
  __device__ void row(int64_t i, const P2& p, const Mat3* a9, const Vec3* a3, Mat3* o9, Vec3* o3, const float* tab) const {
    Quat qh;
    Quat qm = p_mean_quat(a9[0], a3[0], p.k_recip, p.k_recipm1, p.k_c1, p.k_c2, &qh);
    const Vec3 st = a3[1], ps = a3[2];
    Vec3 m;
    m.x = fmaf(p.k_c1, fmaf(p.k_recip, st.x, -p.k_recipm1 * ps.x), p.k_c2 * st.x);
    m.y = fmaf(p.k_c1, fmaf(p.k_recip, st.y, -p.k_recipm1 * ps.y), p.k_c2 * st.y);
    m.z = fmaf(p.k_c1, fmaf(p.k_recip, st.z, -p.k_recipm1 * ps.z), p.k_c2 * st.z);
    if (post_cdf && p.ti != 0) {
      float ang;
      if (post_guide) {
        const GuideRec rec{p.rec.x, __uint_as_float(p.rec.y), __uint_as_float(p.rec.z), __uint_as_float(p.rec.w)};
        ang = igso3_angle_from_record(post_cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, rec, p.d.u);
      } else {
        ang = igso3_angle_from_uniform(post_cdf + (int64_t)p.ti * kCdf, tab + kTabLoc, p.d.u);
      }
      qm = qmul(qm, quat_axis_angle(p.d.axis, ang));
      const Normal4 z = normal4_from_u4(philox4x32_10(key_shift, row_offset + (uint64_t)i));
      const float ns = p.k_sigma * shift_scale;
      m = Vec3{fmaf(ns, z.a, m.x), fmaf(ns, z.b, m.y), fmaf(ns, z.c, m.z)};
    }
    o9[0] = quat_to_mat_unit(qm);
    o3[0] = m;
  }
};

// The shared-t SE(3) reverse step on two rows per thread (rowwise_kernel_cta2): rotation half through the two-lane
// arithmetic of so3d_lanes.cuh, translation half as packed FMAs; the same IEEE operations per row as SE3PStepOp<true>.
#ifndef SO3D_SE3PS2_MINCTAS
#define SO3D_SE3PS2_MINCTAS 5
#endif
template <bool kDevSeed = false>
struct SE3PStep2Op : DevSeedArgs<kDevSeed> {
  SO3D_OP_ARRAYS_S(1, 3, 1, 1, 1)  // in: rot_t | pred_rot, shift_t, pred_shift;  out: rot | shift
  static constexpr int kTab = kTabCdfFloats;
  static constexpr int kMinCtas = SO3D_SE3PS2_MINCTAS;
  static constexpr int kInStages = 1;
  const int64_t* t;
  const float* recip;
  const float* recipm1;
  const float* coef1;
  const float* coef2;
  const float* sigma;
  int64_t T;
  const float* post_cdf;
  const float* loc;
  float shift_scale;
  PhiloxKey key, key_shift;
  uint64_t row_offset;
  __device__ int64_t clamp_t(int64_t ti) const { return ti < 0 ? 0 : (ti >= T ? T - 1 : ti); }
  __device__ void setup(float* tab) const {
    if (post_cdf) stage_cdf(tab, post_cdf + clamp_t(t[0]) * kCdf, loc);
    if (threadIdx.x == 0) {
      const int64_t ti = clamp_t(t[0]);
      tab[kTabScal] = __int_as_float((int)ti);
      tab[kTabScal + 1] = recip[ti];
      tab[kTabScal + 2] = recipm1[ti];
      tab[kTabScal + 3] = coef1[ti];
      tab[kTabScal + 4] = coef2[ti];
      tab[kTabScal + 5] = sigma ? sigma[ti] : 0.f;
      if constexpr (kDevSeed) {
        const uint64_t sd = *this->seed_dev;
        tab[kTabScal + 6] = __uint_as_float((uint32_t)sd);
        tab[kTabScal + 7] = __uint_as_float((uint32_t)(sd >> 32));
      }
    }
  }
  // the rotation and translation blocks of global row r (kDevSeed: from the staged seed)
  __device__ U4 rot_block(uint64_t r, const float* tab) const {
    if constexpr (kDevSeed) return philox4x32_10(staged_seed(tab), r, this->rng_offset);
    else return philox4x32_10(key, r);
  }
  __device__ U4 shift_block(uint64_t r, const float* tab) const {
    if constexpr (kDevSeed) return philox4x32_10(staged_seed(tab), r, this->rng_offset | kShiftStream);
    else return philox4x32_10(key_shift, r);
  }
  __device__ void row2(int64_t i0, const Mat3 (*a9)[2], const Vec3 (*a3)[2], Mat3 (*o9)[2], Vec3 (*o3)[2], const float* tab) const {
    const int ti = __float_as_int(tab[kTabScal]);
    const float k_recip = tab[kTabScal + 1], k_recipm1 = tab[kTabScal + 2], k_c1 = tab[kTabScal + 3], k_c2 = tab[kTabScal + 4],
                k_sigma = tab[kTabScal + 5];
    const Mat3L<L2> x = lanes_of(a9[0][0], a9[0][1]);
    const Vec3L<L2> pred{L2{a3[0][0].x, a3[0][1].x}, L2{a3[0][0].y, a3[0][1].y}, L2{a3[0][0].z, a3[0][1].z}};
    QuatL<L2> qh;
    QuatL<L2> qm = p_mean_quat_l<L2, true>(x, pred, k_recip, k_recipm1, k_c1, k_c2, &qh);
    // translation: m = c1 (recip st - recipm1 ps) + c2 st   (same association as SE3PStepOp::row)
    const Vec3L<L2> st{L2{a3[1][0].x, a3[1][1].x}, L2{a3[1][0].y, a3[1][1].y}, L2{a3[1][0].z, a3[1][1].z}};
    const Vec3L<L2> ps{L2{a3[2][0].x, a3[2][1].x}, L2{a3[2][0].y, a3[2][1].y}, L2{a3[2][0].z, a3[2][1].z}};
    const L2 c1 = bc<L2>(k_c1), c2 = bc<L2>(k_c2), rc = bc<L2>(k_recip), nrm1 = bc<L2>(-k_recipm1);
    Vec3L<L2> m{fma(c1, fma(rc, st.x, mul(nrm1, ps.x)), mul(c2, st.x)), fma(c1, fma(rc, st.y, mul(nrm1, ps.y)), mul(c2, st.y)),
                fma(c1, fma(rc, st.z, mul(nrm1, ps.z)), mul(c2, st.z))};
    if (post_cdf && ti != 0) {
      const uint64_t row = row_offset + (uint64_t)i0;
      const U4 r0 = rot_block(row, tab), r1 = rot_block(row + kT2, tab);
      const Vec3L<L2> axis = sphere_from_uniforms_l(L2{u01(r0.x), u01(r1.x)}, L2{u01(r0.y), u01(r1.y)});
      const L2 ang{shared_row_angle(tab, u01(r0.z)), shared_row_angle(tab, u01(r1.z))};
      qm = qmul_l(qm, quat_axis_angle_l(axis, ang));
      const Normal4 z0 = normal4_from_u4(shift_block(row, tab)), z1 = normal4_from_u4(shift_block(row + kT2, tab));
      const L2 ns = bc<L2>(k_sigma * shift_scale);
      m = Vec3L<L2>{fma(ns, L2{z0.a, z1.a}, m.x), fma(ns, L2{z0.b, z1.b}, m.y), fma(ns, L2{z0.c, z1.c}, m.z)};
    }
    const Mat3L<L2> o = quat_to_mat_unit_l(qm);
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      o9[0][0].m[k] = o.m[k].x;
      o9[0][1].m[k] = o.m[k].y;
    }
    o3[0][0] = Vec3{m.x.x, m.y.x, m.z.x};
    o3[0][1] = Vec3{m.x.y, m.y.y, m.z.y};
  }
};

}  // namespace

// error / device helpers shared with the other translation units of the library (so3d_common.cuh)
namespace so3d_host {
int fail(int code, const char* what) { return ::fail(code, what); }
int check_launch(const char* name) { return ::check_launch(name); }
int sm_count() { return ::sm_count(); }
int current_device() { return ::current_device(); }
}  // namespace so3d_host

// ================================================================================================
// C ABI
// ================================================================================================
extern "C" {

int so3d_version(void) { return SO3D_VERSION; }
const char* so3d_last_error(void) { return g_err; }

#define SO3D_REQUIRE(cond, msg) \
  if (!(cond)) return fail(SO3D_EINVAL, msg)

int so3d_log_f32(const float* R, float* out9, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && out9), "so3d_log_f32: null pointer");
  LogOp op;
  op.in9[0] = R; op.out9[0] = out9;
  return launch_rowwise_pick(op, n, stream, "so3d_log_f32");
}

int so3d_logvec_f32(const float* R, float* out3, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && out3), "so3d_logvec_f32: null pointer");
  LogVecOp op;
  op.in9[0] = R; op.out3[0] = out3;
  return launch_rowwise_pick(op, n, stream, "so3d_logvec_f32", true);
}

int so3d_rmat_to_aa_f32(const float* R, float* axis3, float* angle, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && axis3 && angle), "so3d_rmat_to_aa_f32: null pointer");
  RmatToAaOp op;
  op.in9[0] = R; op.out3[0] = axis3; op.angle = angle;
  return launch_rowwise_pick(op, n, stream, "so3d_rmat_to_aa_f32");
}

int so3d_aa_to_rmat_f32(const float* axis3, const float* angle, float* R, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (axis3 && angle && R), "so3d_aa_to_rmat_f32: null pointer");
  AaToRmatOp op;
  op.in3[0] = axis3; op.angle = angle; op.out9[0] = R;
  return launch_rowwise_pick(op, n, stream, "so3d_aa_to_rmat_f32");
}

int so3d_expvec_f32(const float* v3, float* R, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (v3 && R), "so3d_expvec_f32: null pointer");
  ExpVecOp op;
  op.in3[0] = v3; op.out9[0] = R;
  return launch_rowwise_pick(op, n, stream, "so3d_expvec_f32");
}

int so3d_scale_f32(const float* R, const float* s, int s_stride, float* out, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && s && out), "so3d_scale_f32: null pointer");
  SO3D_REQUIRE(s_stride == 0 || s_stride == 1, "so3d_scale_f32: s_stride must be 0 or 1");
  ScaleOp op;
  op.in9[0] = R; op.s = s; op.s_stride = s_stride; op.out9[0] = out;
  return launch_rowwise_pick(op, n, stream, "so3d_scale_f32");
}

int so3d_quat_to_rmat_f32(const float* q4, float* R, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (q4 && R), "so3d_quat_to_rmat_f32: null pointer");
  QuatToRmatOp op;
  op.q = q4; op.q_vec = aligned16(q4); op.out9[0] = R;
  return launch_rowwise_pick(op, n, stream, "so3d_quat_to_rmat_f32");
}

int so3d_rmat_to_quat_f32(const float* R, float* q4, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && q4), "so3d_rmat_to_quat_f32: null pointer");
  SO3D_REQUIRE(aligned16(q4), "so3d_rmat_to_quat_f32: q4 must be 16-byte aligned");
  RmatToQuatOp op;
  op.in9[0] = R; op.q = q4;
  return launch_rowwise_pick(op, n, stream, "so3d_rmat_to_quat_f32");
}

}  // extern "C"

template <bool TA, bool TB>
static int compose_dispatch(const float* A, int a_stride, const float* B, int b_stride, float* C, int64_t n, void* stream) {
  if (a_stride && b_stride) {
    ComposeOp<TA, TB> op;
    op.in9[0] = A; op.in9[1] = B; op.out9[0] = C;
    return launch_rowwise_pick(op, n, stream, "so3d_compose_f32");
  } else if (!a_stride && b_stride) {
    ComposeSharedOp<TA, TB, true> op;
    op.in9[0] = B; op.shared = A; op.out9[0] = C;
    return launch_rowwise_pick(op, n, stream, "so3d_compose_f32");
  } else if (a_stride && !b_stride) {
    ComposeSharedOp<TA, TB, false> op;
    op.in9[0] = A; op.shared = B; op.out9[0] = C;
    return launch_rowwise_pick(op, n, stream, "so3d_compose_f32");
  }
  return fail(SO3D_EINVAL, "so3d_compose_f32: at most one operand may be shared");
}

extern "C" {

int so3d_compose_f32(const float* A, int a_stride, int trans_a, const float* B, int b_stride, int trans_b, float* C,
                     int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (A && B && C), "so3d_compose_f32: null pointer");
  if (trans_a && trans_b) return compose_dispatch<true, true>(A, a_stride, B, b_stride, C, n, stream);
  if (trans_a) return compose_dispatch<true, false>(A, a_stride, B, b_stride, C, n, stream);
  if (trans_b) return compose_dispatch<false, true>(A, a_stride, B, b_stride, C, n, stream);
  return compose_dispatch<false, false>(A, a_stride, B, b_stride, C, n, stream);
}

int so3d_rmat_dist_f32(const float* A, const float* B, float* out, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (A && B && out), "so3d_rmat_dist_f32: null pointer");
  RmatDistOp op;
  op.in9[0] = A; op.in9[1] = B; op.out = out;
  return launch_rowwise_pick(op, n, stream, "so3d_rmat_dist_f32", true);
}

int so3d_lerp_f32(const float* A, const float* B, const float* w, int w_stride, float* out, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (A && B && w && out), "so3d_lerp_f32: null pointer");
  SO3D_REQUIRE(w_stride == 0 || w_stride == 1, "so3d_lerp_f32: w_stride must be 0 or 1");
  LerpOp op;
  op.in9[0] = A; op.in9[1] = B; op.w = w; op.w_stride = w_stride; op.out9[0] = out;
  return launch_rowwise_pick(op, n, stream, "so3d_lerp_f32");
}

int so3d_log_bwd_f32(const float* R, const float* G9, float* gR, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && G9 && gR), "so3d_log_bwd_f32: null pointer");
  LogBwdOp op;
  op.in9[0] = R; op.in9[1] = G9; op.out9[0] = gR;
  return launch_rowwise_pick(op, n, stream, "so3d_log_bwd_f32");
}

int so3d_aa_to_rmat_bwd_f32(const float* axis3, const float* angle, const float* G9, float* g_axis3, float* g_angle,
                            int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (axis3 && angle && G9 && g_axis3 && g_angle), "so3d_aa_to_rmat_bwd_f32: null pointer");
  AaToRmatBwdOp op;
  op.in9[0] = G9; op.in3[0] = axis3; op.angle = angle; op.out3[0] = g_axis3; op.g_angle = g_angle;
  return launch_rowwise_pick(op, n, stream, "so3d_aa_to_rmat_bwd_f32");
}

int so3d_expvec_bwd_f32(const float* v3, const float* G9, float* g_v3, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (v3 && G9 && g_v3), "so3d_expvec_bwd_f32: null pointer");
  ExpVecBwdOp op;
  op.in9[0] = G9; op.in3[0] = v3; op.out3[0] = g_v3;
  return launch_rowwise_pick(op, n, stream, "so3d_expvec_bwd_f32");
}

int so3d_scale_bwd_f32(const float* R, const float* s, int s_stride, const float* G9, float* gR, float* g_s, int64_t n,
                       void* stream) {
  SO3D_REQUIRE(n == 0 || (R && s && G9 && gR), "so3d_scale_bwd_f32: null pointer");
  SO3D_REQUIRE(s_stride == 0 || s_stride == 1, "so3d_scale_bwd_f32: s_stride must be 0 or 1");
  ScaleBwdOp op;
  op.in9[0] = R; op.in9[1] = G9; op.s = s; op.s_stride = s_stride; op.g_s = g_s; op.out9[0] = gR;
  return launch_rowwise_pick(op, n, stream, "so3d_scale_bwd_f32");
}

}  // extern "C"

template <int kMode>
static int launch_logp_score(const float* R, const float* eps, int eps_stride, float* logp, float* score3, float* dlogf, int64_t n, int L,
                             void* stream) {
  constexpr bool kSeriesMode = LogpScore2Op<kMode>::kSeriesMode;
  if constexpr (kSeriesMode || SO3D_LOGP_PREFETCH) {
    const char* lanes_env = getenv("SO3D_LOGP_LANES");
    if (!(lanes_env && atoi(lanes_env) == 1)) {
      LogpScore2Op<kMode> op2;
      op2.in9[0] = R; op2.eps = eps; op2.eps_stride = eps_stride; op2.logp = logp; op2.dlogf = dlogf; op2.out3[0] = score3;
      op2.L = L; op2.n = n;
      // Resident CTAs per SM of the two-row series kernel, measured on B200 at 2^24 rows (profiles/r06a_series_lanes.jsonl):
      // series / series_pure gain with every resident CTA up to the 6 that fit (series 9.39 ms at 2, 8.66 at 6), series_adaptive
      // (a different trip count per warp) runs fastest at 3 like the one-row kernel (7.02 ms, 7.74 at 6).
      return launch_rowwise_w2(op2, n, stream, "so3d_igso3_logp_score_f32", kMode == kSeriesAdaptive ? 3 : 0);
    }
  }
  LogpScoreOp<kMode> op;
  op.in9[0] = R; op.eps = eps; op.eps_stride = eps_stride; op.logp = logp; op.dlogf = dlogf; op.out3[0] = score3;
  op.L = L;
  // The series streams its constant table through the uniform datapath; measured on B200 it runs fastest with few
  // resident warps (3 CTAs/SM: 1.54e9 evals/s, 8 CTAs/SM: 1.26e9): warps at fewer distinct table positions.
  const int ctas = (kMode == kSeries || kMode == kSeriesAdaptive || kMode == kSeriesPure) ? 3 : 0;
  return launch_rowwise(op, n, stream, "so3d_igso3_logp_score_f32", ctas);
}

extern "C" {

static int check_mode(int mode, int L) {
  if (mode < 0 || mode > 4) return fail(SO3D_EINVAL, "mode must be SO3D_MODE_{SERIES,CLOSED,AUTO,SERIES_ADAPTIVE,SERIES_PURE}");
  if (mode != SO3D_MODE_CLOSED && (L < 1 || L > 2896)) return fail(SO3D_EINVAL, "series truncation L must be in [1, 2896]");
  return 0;
}

int so3d_igso3_density_f32(const float* omega, const float* eps, int eps_stride, float* f, int64_t n, int mode, int L,
                           void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(omega && eps && f, "so3d_igso3_density_f32: null pointer");
  SO3D_REQUIRE(eps_stride == 0 || eps_stride == 1, "eps_stride must be 0 or 1");
  if (int rc = check_mode(mode, L)) return rc;
  const int64_t blocks = (n + 255) / 256;
  const int64_t cap = (int64_t)sm_count() * 8;
  density_kernel<<<(int)(blocks < cap ? blocks : cap), 256, 0, (cudaStream_t)stream>>>(omega, eps, eps_stride, f, n, mode, L);
  return check_launch("so3d_igso3_density_f32");
}

int so3d_igso3_logp_score_f32(const float* R, const float* eps, int eps_stride, float* logp, float* score3, float* dlogf,
                              int64_t n, int mode, int L, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && eps && logp), "so3d_igso3_logp_score_f32: null pointer");
  SO3D_REQUIRE(eps_stride == 0 || eps_stride == 1, "eps_stride must be 0 or 1");
  if (int rc = check_mode(mode, L)) return rc;
  // small batches of the series: one warp per rotation (up to 64 rows per SM -- one full wave of warps -- the
  // one-thread-per-rotation kernel is a handful of warps running 2000-term dependent chains; measured cross-over ~14 000 rows
  // on 148 SMs, profiles/r03m_bench.json; SO3D_SERIES_WARP_ROWS overrides the threshold, 0 disables)
  if (n > 0 && (mode == SO3D_MODE_SERIES || mode == SO3D_MODE_SERIES_ADAPTIVE || mode == SO3D_MODE_SERIES_PURE)) {
    static const int64_t rows_per_sm = [] { const char* e = getenv("SO3D_SERIES_WARP_ROWS"); return e ? (int64_t)atoll(e) : (int64_t)64; }();
    if (n <= rows_per_sm * sm_count()) {
      const int64_t blocks = (n * 32 + 255) / 256;
      const int64_t cap = (int64_t)sm_count() * 8;
      const int grid = (int)(blocks < cap ? blocks : cap);
      if (mode == SO3D_MODE_SERIES_PURE)
        series_warp_kernel<kSeriesPure><<<grid, 256, 0, (cudaStream_t)stream>>>(R, eps, eps_stride, logp, score3, dlogf, n, L);
      else
        series_warp_kernel<kSeries><<<grid, 256, 0, (cudaStream_t)stream>>>(R, eps, eps_stride, logp, score3, dlogf, n, L);
      return check_launch("so3d_igso3_logp_score_f32");
    }
  }
  switch (mode) {
    case SO3D_MODE_SERIES: return launch_logp_score<kSeries>(R, eps, eps_stride, logp, score3, dlogf, n, L, stream);
    case SO3D_MODE_CLOSED: return launch_logp_score<kClosed>(R, eps, eps_stride, logp, score3, dlogf, n, L, stream);
    case SO3D_MODE_AUTO: return launch_logp_score<kAuto>(R, eps, eps_stride, logp, score3, dlogf, n, L, stream);
    case SO3D_MODE_SERIES_PURE: return launch_logp_score<kSeriesPure>(R, eps, eps_stride, logp, score3, dlogf, n, L, stream);
    default: return launch_logp_score<kSeriesAdaptive>(R, eps, eps_stride, logp, score3, dlogf, n, L, stream);
  }
}

int so3d_igso3_logp_bwd_f32(const float* R, const float* dlogf, const float* gout, float* gR, int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (R && dlogf && gout && gR), "so3d_igso3_logp_bwd_f32: null pointer");
  LogpBwdOp op;
  op.in9[0] = R; op.dlogf = dlogf; op.gout = gout; op.out9[0] = gR;
  return launch_rowwise_pick(op, n, stream, "so3d_igso3_logp_bwd_f32");
}

int so3d_igso3_cdf_table_f32(const float* eps, int64_t rows, const float* grid_loc, const float* haar_w, float* trap_out,
                             int quirks, void* stream) {
  SO3D_REQUIRE(rows >= 0, "negative rows");
  if (rows == 0) return 0;
  SO3D_REQUIRE(eps && grid_loc && haar_w && trap_out, "so3d_igso3_cdf_table_f32: null pointer");
  SO3D_REQUIRE(rows <= 0x7fffffff, "so3d_igso3_cdf_table_f32: too many rows");
  cdf_table_kernel<<<(int)rows, 256, 0, (cudaStream_t)stream>>>(eps, grid_loc, haar_w, trap_out, quirks);
  return check_launch("so3d_igso3_cdf_table_f32");
}

}  // extern "C"

template <bool kShared>
static int launch_sample(const float* cdf, const uint32_t* guide, const float* loc, int64_t rows, const int64_t* row_idx, int64_t row,
                         const float* u, const float* axes3, uint64_t seed, uint64_t rng_offset, uint64_t row_offset, const float* mean,
                         int mean_stride, float* R, float* angle, float* axis3, int64_t n, void* stream) {
  SampleOp<kShared> op;
  op.out9[0] = R; op.out3[0] = axis3;
  op.cdf = cdf; op.guide = guide; op.loc = loc; op.row_idx = row_idx; op.shared_row = row; op.rows = rows; op.u_in = u; op.axes_in = axes3;
  op.key = make_philox_key(seed, rng_offset); op.key_shift = make_philox_key(seed, rng_offset | kShiftStream); op.row_offset = row_offset; op.mean = mean; op.mean_stride = mean_stride; op.angle_out = angle;
  // (prefetch hooks for the per-row table rows measured no gain here, 0.2329 ms either way, r05g: the kernel is bound by its 48 B/row of writes)
  return launch_rowwise_pick(op, n, stream, "so3d_igso3_sample_f32");
}

template <bool kExtra, bool kDevSeed = false, bool kNoiseOut = kExtra>
static int launch_q_sample(const float* x0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac, int64_t T, const float* cdf,
                           const uint32_t* guide, const float* loc, uint64_t seed, uint64_t rng_offset, uint64_t row_offset, float* x_t,
                           float* target3, float* noise, float* score3, int64_t n, void* stream, const uint64_t* seed_dev = nullptr) {
  // two rows per thread with packed FP32 on the warp-autonomous schedule (SO3D_QS_LANES=1 selects the one-row kernel for A/B runs)
  // (read per call: the cross-kernel parity test switches it; the variant that also writes the noise matrix would spill
  // at 128 registers and stays on the one-row kernel)
  const char* lanes_env = getenv("SO3D_QS_LANES");
  const bool one_lane = kNoiseOut || (lanes_env ? atoi(lanes_env) == 1 : !SO3D_QS_LANES_DEFAULT2);
  auto fill = [&](auto& op) {
    op.seed_dev = seed_dev; op.rng_offset = rng_offset;
    op.in9[0] = x0; op.out9[0] = x_t; op.out3[0] = target3;
    if (kNoiseOut) op.out9[kNoiseOut ? 1 : 0] = noise;
    if (kExtra) op.out3[kExtra ? 1 : 0] = score3;
    op.t = t; op.sqrt_ac = sqrt_ac; op.sqrt_1m_ac = sqrt_1m_ac; op.T = T; op.cdf = cdf; op.guide = guide; op.loc = loc;
    op.key = make_philox_key(seed, rng_offset); op.key_shift = make_philox_key(seed, rng_offset | kShiftStream); op.row_offset = row_offset;
  };
  if constexpr (!kNoiseOut) {
    if (!one_lane) {
      QSample2Op<kExtra, kDevSeed, kNoiseOut> op2;
      fill(op2);
      return launch_rowwise_w2(op2, n, stream, "so3d_q_sample_f32");
    }
  }
  QSampleOp<kExtra, kDevSeed, kNoiseOut> op;
  fill(op);
  return launch_rowwise(op, n, stream, "so3d_q_sample_f32");
}

template <bool kSharedT, bool kX0, bool kDevSeed = false>
static int launch_p_step(const float* x_t, const float* pred3, const int64_t* t, const float* recip, const float* recipm1,
                         const float* coef1, const float* coef2, int64_t T, const float* post_cdf, const uint32_t* post_guide,
                         const float* loc, uint64_t seed, uint64_t rng_offset, uint64_t row_offset, float* out, float* x0_hat_out,
                         int64_t n, void* stream, const uint64_t* seed_dev = nullptr) {
  if constexpr (kSharedT && !kX0) {
    // the hot shared-t step: two rows per thread with packed FP32 (SO3D_PSTEP_LANES=1 selects the one-row kernel for A/B runs)
    static const bool one_lane = [] { const char* e = getenv("SO3D_PSTEP_LANES"); return e && atoi(e) == 1; }();
    static const bool w2_engine = [] { const char* e = getenv("SO3D_PSTEP_ENGINE"); return e && strcmp(e, "w2") == 0; }();
    if (!one_lane && post_cdf && w2_engine) {
      PStep2wOp<kDevSeed> op2;
      op2.seed_dev = seed_dev;
      op2.in9[0] = x_t; op2.in3[0] = pred3; op2.out9[0] = out;
      op2.t = t; op2.recip = recip; op2.recipm1 = recipm1; op2.coef1 = coef1; op2.coef2 = coef2; op2.T = T;
      op2.post_cdf = post_cdf; op2.loc = loc; op2.seed = seed; op2.rng_offset = rng_offset; op2.row_offset = row_offset;
      return launch_rowwise_w2(op2, n, stream, "so3d_p_sample_f32");
    }
    if (!one_lane && post_cdf) {
      PStep2Op<kDevSeed> op2;
      op2.seed_dev = seed_dev;
      op2.in9[0] = x_t; op2.in3[0] = pred3; op2.out9[0] = out;
      op2.t = t; op2.recip = recip; op2.recipm1 = recipm1; op2.coef1 = coef1; op2.coef2 = coef2; op2.T = T;
      op2.post_cdf = post_cdf; op2.loc = loc; op2.seed = seed; op2.rng_offset = rng_offset; op2.row_offset = row_offset;
      return launch_rowwise2(op2, n, stream, "so3d_p_sample_f32");
    }
  }
  if constexpr (!kSharedT && !kX0 && SO3D_PS_PREFETCH) {
    // per-row t: two rows per thread on the warp-autonomous two-row schedule (SO3D_PS_LANES=1: the one-row kernel; read per call
    // for the cross-kernel parity test)
    const char* lanes_env = getenv("SO3D_PS_LANES");
    if (!(lanes_env && atoi(lanes_env) == 1)) {
      PStepRows2Op<kDevSeed> op2;
      op2.seed_dev = seed_dev;
      op2.in9[0] = x_t; op2.in3[0] = pred3; op2.out9[0] = out;
      op2.t = t; op2.recip = recip; op2.recipm1 = recipm1; op2.coef1 = coef1; op2.coef2 = coef2; op2.T = T;
      op2.post_cdf = post_cdf; op2.post_guide = post_guide; op2.loc = loc; op2.seed = seed; op2.rng_offset = rng_offset; op2.row_offset = row_offset;
      return launch_rowwise_w2(op2, n, stream, "so3d_p_sample_f32");
    }
  }
  PStepOp<kSharedT, kX0, kDevSeed> op;
  op.seed_dev = seed_dev;
  op.in9[0] = x_t; op.in3[0] = pred3; op.out9[0] = out;
  if (kX0) op.out9[kX0 ? 1 : 0] = x0_hat_out;
  op.t = t; op.recip = recip; op.recipm1 = recipm1; op.coef1 = coef1; op.coef2 = coef2; op.T = T;
  op.post_cdf = post_cdf; op.post_guide = post_guide; op.loc = loc; op.seed = seed; op.rng_offset = rng_offset; op.row_offset = row_offset;
  return launch_rowwise(op, n, stream, "so3d_p_sample_f32");
}

extern "C" {

int so3d_igso3_sample_f32(const float* cdf, const uint32_t* guide, const float* loc, int64_t rows, const int64_t* row_idx, int64_t row,
                          const float* u, const float* axes3, uint64_t seed, uint64_t rng_offset, uint64_t row_offset,
                          const float* mean, int mean_stride, float* R, float* angle, float* axis3, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(cdf && loc && R, "so3d_igso3_sample_f32: null pointer");
  SO3D_REQUIRE(rows > 0, "so3d_igso3_sample_f32: empty table");
  SO3D_REQUIRE(row_idx || (row >= 0 && row < rows), "so3d_igso3_sample_f32: row out of range");
  SO3D_REQUIRE(mean_stride == 0 || mean_stride == 1, "mean_stride must be 0 or 1");
  if (row_idx)
    return launch_sample<false>(cdf, guide, loc, rows, row_idx, 0, u, axes3, seed, rng_offset, row_offset, mean, mean_stride, R, angle, axis3, n, stream);
  return launch_sample<true>(cdf, guide, loc, rows, nullptr, row, u, axes3, seed, rng_offset, row_offset, mean, mean_stride, R, angle, axis3, n, stream);
}

int so3d_igso3_sample_exact_f32(const float* eps, int eps_stride, const float* u, const float* axes3, uint64_t seed, uint64_t rng_offset,
                                uint64_t row_offset, const float* mean, int mean_stride, float* R, float* angle, float* axis3, int64_t n,
                                void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(eps && R, "so3d_igso3_sample_exact_f32: null pointer");
  SO3D_REQUIRE(eps_stride == 0 || eps_stride == 1, "eps_stride must be 0 or 1");
  SO3D_REQUIRE(mean_stride == 0 || mean_stride == 1, "mean_stride must be 0 or 1");
  SampleExactOp op;
  op.out9[0] = R; op.out3[0] = axis3;
  op.eps = eps; op.eps_stride = eps_stride; op.u_in = u; op.axes_in = axes3;
  op.key = make_philox_key(seed, rng_offset); op.row_offset = row_offset; op.mean = mean; op.mean_stride = mean_stride; op.angle_out = angle;
  return launch_rowwise_pick(op, n, stream, "so3d_igso3_sample_exact_f32");
}

int so3d_igso3_rsample_bwd_f32(const float* eps, int eps_stride, const float* angle, const float* axis3, const float* mean,
                               int mean_stride, const float* G9, const float* u, uint64_t seed, uint64_t rng_offset,
                               uint64_t row_offset, float* g_eps, float* g_mean9, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(eps && angle && axis3 && G9 && g_eps, "so3d_igso3_rsample_bwd_f32: null pointer");
  SO3D_REQUIRE(eps_stride == 0 || eps_stride == 1, "eps_stride must be 0 or 1");
  SO3D_REQUIRE(mean_stride == 0 || mean_stride == 1, "mean_stride must be 0 or 1");
  RsampleBwdOp op;
  op.in9[0] = G9; op.in3[0] = axis3; op.out9[0] = g_mean9;
  op.eps = eps; op.eps_stride = eps_stride; op.angle = angle; op.mean = mean; op.mean_stride = mean_stride;
  op.u_in = u; op.key = make_philox_key(seed, rng_offset); op.row_offset = row_offset; op.g_eps = g_eps;
  return launch_rowwise_pick(op, n, stream, "so3d_igso3_rsample_bwd_f32");
}

int so3d_q_sample_f32(const float* x0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac, int64_t T,
                      const float* cdf, const uint32_t* guide, const float* loc, uint64_t seed, uint64_t rng_offset,
                      uint64_t row_offset, float* x_t, float* target3, float* noise, float* score3, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(x0 && t && sqrt_ac && sqrt_1m_ac && cdf && loc && x_t, "so3d_q_sample_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_q_sample_f32: T must be positive");
  if (score3 && !noise)
    return launch_q_sample<true, false, false>(x0, t, sqrt_ac, sqrt_1m_ac, T, cdf, guide, loc, seed, rng_offset, row_offset, x_t, target3, nullptr, score3, n,
                                               stream);
  if (noise || score3)
    return launch_q_sample<true>(x0, t, sqrt_ac, sqrt_1m_ac, T, cdf, guide, loc, seed, rng_offset, row_offset, x_t, target3, noise, score3, n, stream);
  return launch_q_sample<false>(x0, t, sqrt_ac, sqrt_1m_ac, T, cdf, guide, loc, seed, rng_offset, row_offset, x_t, target3, noise, score3, n, stream);
}

int so3d_q_sample_dseed_f32(const float* x0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac, int64_t T, const float* cdf,
                            const uint32_t* guide, const float* loc, const uint64_t* seed_dev, uint64_t rng_offset, uint64_t row_offset,
                            float* x_t, float* target3, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(x0 && t && sqrt_ac && sqrt_1m_ac && cdf && loc && x_t && seed_dev, "so3d_q_sample_dseed_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_q_sample_dseed_f32: T must be positive");
  return launch_q_sample<false, true>(x0, t, sqrt_ac, sqrt_1m_ac, T, cdf, guide, loc, 0, rng_offset, row_offset, x_t, target3, nullptr, nullptr, n,
                                      stream, seed_dev);
}

int so3d_q_sample_given_f32(const float* x0, const int64_t* t, const float* sqrt_ac, int64_t T, const float* noise, float* x_t,
                            int64_t n, void* stream) {
  SO3D_REQUIRE(n == 0 || (x0 && t && sqrt_ac && noise && x_t), "so3d_q_sample_given_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_q_sample_given_f32: T must be positive");
  QSampleGivenOp op;
  op.in9[0] = x0; op.in9[1] = noise; op.out9[0] = x_t; op.t = t; op.sqrt_ac = sqrt_ac; op.T = T;
  return launch_rowwise_pick(op, n, stream, "so3d_q_sample_given_f32");
}

int so3d_bingham_sample_f32(const float* scale_tril16, const float* z4, uint64_t seed, uint64_t rng_offset, uint64_t row_offset,
                            float* q4, float* R, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(scale_tril16 && (q4 || R), "so3d_bingham_sample_f32: scale_tril16 and at least one output are required");
  SO3D_REQUIRE(!q4 || aligned16(q4), "so3d_bingham_sample_f32: q4 must be 16-byte aligned");
  BinghamOp op;
  op.out9[0] = R; op.tril = scale_tril16; op.z_in = z4; op.z_vec = aligned16(z4); op.q_out = q4;
  op.key = make_philox_key(seed, rng_offset); op.key_shift = make_philox_key(seed, rng_offset | kShiftStream); op.row_offset = row_offset;
  return launch_rowwise_pick(op, n, stream, "so3d_bingham_sample_f32");
}

int so3d_igso3_cdf_guide(const float* cdf, int64_t rows, uint32_t* guide_out, void* stream) {
  SO3D_REQUIRE(rows >= 0, "negative rows");
  if (rows == 0) return 0;
  SO3D_REQUIRE(cdf && guide_out, "so3d_igso3_cdf_guide: null pointer");
  SO3D_REQUIRE(aligned16(guide_out), "so3d_igso3_cdf_guide: guide_out must be 16-byte aligned");
  SO3D_REQUIRE(rows <= 0x7fffffff, "so3d_igso3_cdf_guide: too many rows");
  cdf_guide_kernel<<<(int)rows, kTile, 0, (cudaStream_t)stream>>>(cdf, guide_out);
  return check_launch("so3d_igso3_cdf_guide");
}

int so3d_p_sample_f32(const float* x_t, const float* pred3, const int64_t* t, int t_stride, const float* recip,
                      const float* recipm1, const float* coef1, const float* coef2, int64_t T, const float* post_cdf,
                      const uint32_t* post_guide, const float* loc, uint64_t seed, uint64_t rng_offset, uint64_t row_offset,
                      float* out, float* x0_hat_out, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(x_t && pred3 && t && recip && recipm1 && coef1 && coef2 && out, "so3d_p_sample_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_p_sample_f32: T must be positive");
  SO3D_REQUIRE(t_stride == 0 || t_stride == 1, "t_stride must be 0 or 1");
  SO3D_REQUIRE(!post_cdf || loc, "so3d_p_sample_f32: loc required with post_cdf");
#define SO3D_PSTEP(S, X) \
  launch_p_step<S, X>(x_t, pred3, t, recip, recipm1, coef1, coef2, T, post_cdf, post_guide, loc, seed, rng_offset, row_offset, out, x0_hat_out, n, stream)
  if (t_stride == 0) return x0_hat_out ? SO3D_PSTEP(true, true) : SO3D_PSTEP(true, false);
  return x0_hat_out ? SO3D_PSTEP(false, true) : SO3D_PSTEP(false, false);
#undef SO3D_PSTEP
}

int so3d_p_sample_dseed_f32(const float* x_t, const float* pred3, const int64_t* t, const float* recip, const float* recipm1,
                            const float* coef1, const float* coef2, int64_t T, const float* post_cdf, const float* loc,
                            const uint64_t* seed_dev, uint64_t rng_offset, uint64_t row_offset, float* out, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(x_t && pred3 && t && recip && recipm1 && coef1 && coef2 && out && post_cdf && loc && seed_dev, "so3d_p_sample_dseed_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_p_sample_dseed_f32: T must be positive");
  return launch_p_step<true, false, true>(x_t, pred3, t, recip, recipm1, coef1, coef2, T, post_cdf, nullptr, loc, 0, rng_offset, row_offset, out,
                                          nullptr, n, stream, seed_dev);
}

}  // extern "C"

template <bool kSharedT, bool kDevSeed = false>
static int launch_se3_p_step(const float* rot_t, const float* shift_t, const float* pred_rot3, const float* pred_shift3, const int64_t* t,
                             const float* recip, const float* recipm1, const float* coef1, const float* coef2, const float* sigma, int64_t T,
                             const float* post_cdf, const uint32_t* post_guide, const float* loc, float shift_scale, uint64_t seed,
                             uint64_t rng_offset, uint64_t row_offset, float* rot_out, float* shift_out, int64_t n, void* stream,
                             const uint64_t* seed_dev = nullptr) {
  const char* name = kDevSeed ? "so3d_se3_p_sample_dseed_f32" : "so3d_se3_p_sample_f32";
  auto fill = [&](auto& op) {
    if constexpr (kDevSeed) op.seed_dev = seed_dev, op.rng_offset = rng_offset;
    op.in9[0] = rot_t; op.in3[0] = pred_rot3; op.in3[1] = shift_t; op.in3[2] = pred_shift3; op.out9[0] = rot_out; op.out3[0] = shift_out;
    op.t = t; op.recip = recip; op.recipm1 = recipm1; op.coef1 = coef1; op.coef2 = coef2; op.sigma = sigma; op.T = T;
    op.post_cdf = post_cdf; op.loc = loc; op.shift_scale = shift_scale;
    op.key = make_philox_key(seed, rng_offset); op.key_shift = make_philox_key(seed, rng_offset | kShiftStream); op.row_offset = row_offset;
  };
  if constexpr (kSharedT) {
    // the shared-t step with noise: two rows per thread by default (SO3D_SE3_PSTEP_LANES=1 selects the one-row kernel, A/B aid)
    static const bool one_lane = [] { const char* e = getenv("SO3D_SE3_PSTEP_LANES"); return e && atoi(e) == 1; }();
    if (!one_lane && post_cdf) {
      SE3PStep2Op<kDevSeed> op;
      fill(op);
      return launch_rowwise2(op, n, stream, name);
    }
  }
  SE3PStepOp<kSharedT, kDevSeed> op;
  fill(op);
  op.post_guide = post_guide;
  if constexpr (!kSharedT) {  // per-row t (r05d, r05f)
    if constexpr (SO3D_SE3PS_PREFETCH) return launch_rowwise_pick_pre(op, n, stream, name, SO3D_SE3PS_ROWS_TWO != 0);
    else return launch_rowwise_pick(op, n, stream, name, SO3D_SE3PS_ROWS_TWO != 0);
  }
  return launch_rowwise(op, n, stream, name);
}

template <bool kDevSeed>
static int launch_se3_q_sample(const float* rot0, const float* shift0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac,
                               int64_t T, const float* cdf, const uint32_t* guide, const float* loc, float shift_scale, uint64_t seed,
                               uint64_t rng_offset, uint64_t row_offset, float* rot_t, float* shift_t, float* target_rot3,
                               float* target_shift3, int64_t n, void* stream, const uint64_t* seed_dev = nullptr) {
  const char* name = kDevSeed ? "so3d_se3_q_sample_dseed_f32" : "so3d_se3_q_sample_f32";
  auto fill = [&](auto& op) {
    if constexpr (kDevSeed) op.seed_dev = seed_dev, op.rng_offset = rng_offset;
    op.in9[0] = rot0; op.in3[0] = shift0; op.out9[0] = rot_t; op.out3[0] = target_rot3; op.out3[1] = shift_t; op.out3[2] = target_shift3;
    op.t = t; op.sqrt_ac = sqrt_ac; op.sqrt_1m_ac = sqrt_1m_ac; op.T = T; op.cdf = cdf; op.guide = guide; op.loc = loc;
    op.shift_scale = shift_scale; op.key = make_philox_key(seed, rng_offset); op.key_shift = make_philox_key(seed, rng_offset | kShiftStream); op.row_offset = row_offset;
  };
#if SO3D_SE3QS_PREFETCH
  // Two rows per thread with per-warp input slices: 0.424 -> 0.412 ms (r04k; with the CTA-wide input ring it was no faster,
  // r04f/r04g).  SO3D_SE3_QS_LANES=1 selects the one-row kernel (cross-kernel parity test).
  const char* lanes_env = getenv("SO3D_SE3_QS_LANES");
  if (!(lanes_env && atoi(lanes_env) == 1)) {
    SE3QSample2Op<kDevSeed> op2;
    fill(op2);
    return launch_rowwise_w2(op2, n, stream, name);
  }
#endif
  SE3QSampleOp<kDevSeed> op;
  fill(op);
  return launch_rowwise(op, n, stream, name);
}

extern "C" {

int so3d_se3_q_sample_f32(const float* rot0, const float* shift0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac,
                          int64_t T, const float* cdf, const uint32_t* guide, const float* loc, float shift_scale, uint64_t seed,
                          uint64_t rng_offset, uint64_t row_offset, float* rot_t, float* shift_t, float* target_rot3,
                          float* target_shift3, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(rot0 && shift0 && t && sqrt_ac && sqrt_1m_ac && cdf && loc && rot_t && shift_t, "so3d_se3_q_sample_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_se3_q_sample_f32: T must be positive");
  SO3D_REQUIRE(rng_offset < kShiftStream, "so3d_se3_q_sample_f32: rng_offset must be below 2^63");
  return launch_se3_q_sample<false>(rot0, shift0, t, sqrt_ac, sqrt_1m_ac, T, cdf, guide, loc, shift_scale, seed, rng_offset, row_offset, rot_t,
                                    shift_t, target_rot3, target_shift3, n, stream);
}

int so3d_se3_q_sample_dseed_f32(const float* rot0, const float* shift0, const int64_t* t, const float* sqrt_ac, const float* sqrt_1m_ac,
                                int64_t T, const float* cdf, const uint32_t* guide, const float* loc, float shift_scale,
                                const uint64_t* seed_dev, uint64_t rng_offset, uint64_t row_offset, float* rot_t, float* shift_t,
                                float* target_rot3, float* target_shift3, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(rot0 && shift0 && t && sqrt_ac && sqrt_1m_ac && cdf && loc && rot_t && shift_t && seed_dev,
               "so3d_se3_q_sample_dseed_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_se3_q_sample_dseed_f32: T must be positive");
  SO3D_REQUIRE(rng_offset < kShiftStream, "so3d_se3_q_sample_dseed_f32: rng_offset must be below 2^63");
  return launch_se3_q_sample<true>(rot0, shift0, t, sqrt_ac, sqrt_1m_ac, T, cdf, guide, loc, shift_scale, 0, rng_offset, row_offset, rot_t,
                                   shift_t, target_rot3, target_shift3, n, stream, seed_dev);
}

int so3d_se3_p_sample_f32(const float* rot_t, const float* shift_t, const float* pred_rot3, const float* pred_shift3, const int64_t* t,
                          int t_stride, const float* recip, const float* recipm1, const float* coef1, const float* coef2,
                          const float* sigma, int64_t T, const float* post_cdf, const uint32_t* post_guide, const float* loc,
                          float shift_scale, uint64_t seed, uint64_t rng_offset, uint64_t row_offset, float* rot_out, float* shift_out,
                          int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(rot_t && shift_t && pred_rot3 && pred_shift3 && t && recip && recipm1 && coef1 && coef2 && rot_out && shift_out,
               "so3d_se3_p_sample_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_se3_p_sample_f32: T must be positive");
  SO3D_REQUIRE(t_stride == 0 || t_stride == 1, "t_stride must be 0 or 1");
  SO3D_REQUIRE(!post_cdf || (loc && sigma), "so3d_se3_p_sample_f32: loc and sigma required with post_cdf");
  SO3D_REQUIRE(rng_offset < kShiftStream, "so3d_se3_p_sample_f32: rng_offset must be below 2^63");
  if (t_stride == 0)
    return launch_se3_p_step<true>(rot_t, shift_t, pred_rot3, pred_shift3, t, recip, recipm1, coef1, coef2, sigma, T, post_cdf, post_guide, loc,
                                   shift_scale, seed, rng_offset, row_offset, rot_out, shift_out, n, stream);
  return launch_se3_p_step<false>(rot_t, shift_t, pred_rot3, pred_shift3, t, recip, recipm1, coef1, coef2, sigma, T, post_cdf, post_guide, loc,
                                  shift_scale, seed, rng_offset, row_offset, rot_out, shift_out, n, stream);
}

int so3d_se3_p_sample_dseed_f32(const float* rot_t, const float* shift_t, const float* pred_rot3, const float* pred_shift3, const int64_t* t,
                                const float* recip, const float* recipm1, const float* coef1, const float* coef2, const float* sigma,
                                int64_t T, const float* post_cdf, const float* loc, float shift_scale, const uint64_t* seed_dev,
                                uint64_t rng_offset, uint64_t row_offset, float* rot_out, float* shift_out, int64_t n, void* stream) {
  SO3D_REQUIRE(n >= 0, "negative n");
  if (n == 0) return 0;
  SO3D_REQUIRE(rot_t && shift_t && pred_rot3 && pred_shift3 && t && recip && recipm1 && coef1 && coef2 && sigma && post_cdf && loc && seed_dev &&
                   rot_out && shift_out,
               "so3d_se3_p_sample_dseed_f32: null pointer");
  SO3D_REQUIRE(T > 0, "so3d_se3_p_sample_dseed_f32: T must be positive");
  SO3D_REQUIRE(rng_offset < kShiftStream, "so3d_se3_p_sample_dseed_f32: rng_offset must be below 2^63");
  return launch_se3_p_step<true, true>(rot_t, shift_t, pred_rot3, pred_shift3, t, recip, recipm1, coef1, coef2, sigma, T, post_cdf, nullptr, loc,
                                       shift_scale, 0, rng_offset, row_offset, rot_out, shift_out, n, stream, seed_dev);
}

}  // extern "C"
