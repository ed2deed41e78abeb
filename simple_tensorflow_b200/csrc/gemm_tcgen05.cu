// MatMul / BatchMatMul core for sm_100a: persistent, warp-specialised tcgen05 GEMM.
//
//   C[b][M,N] = op(A[b]) * op(B[b])       fp32 I/O on kind::tf32, bf16 I/O on kind::f16,
//                                          fp32 accumulation in TMEM in both cases.
//
// Replaces the reference's GPU path  LaunchMatMul<GPUDevice,T,true>::launch -> Stream::ThenBlasGemm
// (tensorflow/core/kernels/matmul_op.cc:162-203) and LaunchBatchMatMul<GPUDevice>
// (tensorflow/core/kernels/batch_matmul_op_impl.h:297-363).  All four transpose_a/transpose_b
// combinations are served without any data movement: a row-major [rows,K] operand is "K-major",
// a row-major [K,rows] operand is "MN-major"; both are legal tcgen05 shared-memory layouts for
// tf32 and bf16 (instruction-descriptor bits 15/16).
//
// CTA layout (192 threads, one CTA per SM, persistent over output tiles):
//   warp 0      : TMA producer  (cp.async.bulk.tensor -> 128B-swizzled smem ring, mbarrier tx)
//   warp 1      : TMEM allocator + tcgen05.mma issuer (the whole warp runs the loop, one elected
//                 lane issues each instruction)
//   warps 2..5  : epilogue (tcgen05.ld TMEM -> registers -> fused tail -> 128B-swizzled smem
//                 staging -> TMA store; direct global stores for outputs TMA cannot address)
// Pipelines: smem full/empty ring (kStages), TMEM accumulator full/empty (2 stages) so the
// epilogue of tile i overlaps the main loop of tile i+1.  Split-K partials go to an fp32 scratch
// buffer and are summed in ascending split order by a second, ordered reduction kernel.
#include "b200_ptx.cuh"
#include "b200_internal.h"

#include <cuda_bf16.h>
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <type_traits>

namespace b200 {

constexpr int kBM = 128;          // tile rows  (UMMA M, cta_group::1)
constexpr int kSwizzleBytes = 128;
constexpr int kGemmThreads = 192;
// Epilogue staging: 4 warps x 2 buffers x (32 rows x 128 B), 128B-swizzled, drained by TMA stores.
constexpr int kEpiBufBytes = 32 * kSwizzleBytes;
constexpr int kEpiStageBytes = 4 * 2 * kEpiBufBytes;  // store staging
constexpr int kFeatBufs = 4;                          // feature tiles in flight per epilogue warp
constexpr int kEpiFeatBytes = 4 * kFeatBufs * kEpiBufBytes;  // ReluGrad-features / bias staging

template <typename T>
struct GemmTraits;
template <>
struct GemmTraits<float> {
  static constexpr int kBK = 32;       // 128 B of K per smem row
  static constexpr int kUmmaK = 8;     // tf32: 32 B per instruction
  static constexpr uint32_t kFormat = 2;  // TF32
  static constexpr CUtensorMapDataType kTmaType = CU_TENSOR_MAP_DATA_TYPE_FLOAT32;
};
template <>
struct GemmTraits<__nv_bfloat16> {
  static constexpr int kBK = 64;
  static constexpr int kUmmaK = 16;
  static constexpr uint32_t kFormat = 1;  // BF16
  static constexpr CUtensorMapDataType kTmaType = CU_TENSOR_MAP_DATA_TYPE_BFLOAT16;
};

// kCtas = 1: one CTA computes a 128 x BN tile (tcgen05 cta_group::1).
// kCtas = 2: a CTA PAIR (cluster of 2, the two SMs of a TPC) computes a 256 x BN tile with
//            cta_group::2 MMAs: each CTA stages its own 128 rows of A and its own BN/2 columns of
//            B, so the per-SM L2->smem operand traffic per FLOP halves compared with kCtas = 1
//            (the main loop is L2-fabric bound, see profiles/).
template <int BN, int kCtas>
constexpr int gemm_stages() {
  // stage = A (16 KiB) + B (BN / kCtas rows of 128 B)
  // The main loop is L2-bandwidth bound (~54 GB/s per SM x ~1 us latency = 54 KB in flight), so
  // 4 stages of 32 KiB are plenty; the smem saved feeds the epilogue's prefetch buffers.
  return (BN / kCtas) >= 256 ? 2 : ((BN / kCtas) >= 128 ? 4 : 5);
}
template <int BN, int kCtas>
constexpr size_t gemm_smem_bytes() {
  return static_cast<size_t>(gemm_stages<BN, kCtas>()) *
             (kBM * kSwizzleBytes + (BN / kCtas) * kSwizzleBytes) +
         kEpiStageBytes + kEpiFeatBytes + 1024 + 256;
}

static int plan_splits(long long tiles, int num_kb, int units);

struct GemmShape {
  int M, N, K, batch;
  int ldc;            // elements
  long long strideC;  // elements between batches
  int splits;         // split-K factor (1 = none)
  int kb_per_split;   // K blocks per split
  float* partial;     // [splits][batch][M][N] fp32 partial sums when splits > 1
  int a_map4d, b_map4d;  // MN-major operand described by a 4-D map: one TMA per stage
  // implicit-GEMM convolution A operand (conv_a != 0): K blocks enumerate (filter tap, channel block)
  int conv_a, cv_OW, cv_OH, cv_sh, cv_sw, cv_pt, cv_pl, cv_S, cv_C, cv_cblocks, cv_taps;
  // epilogue
  int tma_store;         // 1: stage through smem and TMA-store via tmapC (C or the partial buffer)
  const void* bias;      // optional fused BiasAdd: + bias[col]      (element type TOut)
  int relu;              // optional fused Relu:     max(x, 0)
  const void* relu_grad_features;  // optional fused ReluGrad: x * (features[row, col] > 0)
  int ld_features;       // leading dimension of features (elements)
  int feat_tma;          // 1: features are fetched by TMA through tmapF (prefetched, coalesced)
  int bias_vec;          // 1: bias pointer is 16-byte aligned (vector loads)
  // B200TF_GEMM_TRACE=1 (debug): %globaltimer at the phase boundaries of the first CTA
  // (slots 0-8) and entry / exit of the last CTA (slots 9, 10)
  unsigned long long* trace;
};
__device__ __forceinline__ void trace_mark(const GemmShape& s, int slot, bool last_cta = false) {
  if (s.trace != nullptr && blockIdx.x == (last_cta ? gridDim.x - 1 : 0)) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    s.trace[slot] = t;
  }
}

// One GEMM of a launch: operand maps, output (or partial-buffer) store map, ReluGrad-feature map.
template <typename TOut>
struct GemmProblem {
  CUtensorMap tmapA, tmapB, tmapC, tmapF;
  TOut* C;
  GemmShape s;
};
// kNP = 1: one GEMM.  kNP = 2: two independent GEMMs with the same tile config in one persistent
// launch (a dense layer's dX and dW); the flat work list holds the `first_work` items of problem
// `first`, then those of the other one.
template <typename TOut, int kNP>
struct GemmParams {
  GemmProblem<TOut> p[kNP];
  int first, first_work;
};

__device__ __forceinline__ void store_row32(float* dst, const uint32_t (&v)[32], int ncols,
                                            bool vec_ok) {
  if (vec_ok && ncols == 32) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float4 f = make_float4(__uint_as_float(v[4 * j]), __uint_as_float(v[4 * j + 1]),
                             __uint_as_float(v[4 * j + 2]), __uint_as_float(v[4 * j + 3]));
      reinterpret_cast<float4*>(dst)[j] = f;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < ncols) dst[j] = __uint_as_float(v[j]);
  }
}
__device__ __forceinline__ void store_row32(__nv_bfloat16* dst, const uint32_t (&v)[32],
                                            int ncols, bool vec_ok) {
  if (vec_ok && ncols == 32) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint4 p;
      __nv_bfloat162 h;
      h = __floats2bfloat162_rn(__uint_as_float(v[8 * j]), __uint_as_float(v[8 * j + 1]));
      p.x = *reinterpret_cast<uint32_t*>(&h);
      h = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 2]), __uint_as_float(v[8 * j + 3]));
      p.y = *reinterpret_cast<uint32_t*>(&h);
      h = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 4]), __uint_as_float(v[8 * j + 5]));
      p.z = *reinterpret_cast<uint32_t*>(&h);
      h = __floats2bfloat162_rn(__uint_as_float(v[8 * j + 6]), __uint_as_float(v[8 * j + 7]));
      p.w = *reinterpret_cast<uint32_t*>(&h);
      reinterpret_cast<uint4*>(dst)[j] = p;
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j)
      if (j < ncols) dst[j] = __float2bfloat16_rn(__uint_as_float(v[j]));
  }
}

__device__ __forceinline__ float ld_as_float(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld_as_float(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <typename TOut>
__host__ __device__ constexpr int nvals_max() {
  return kSwizzleBytes / (int)sizeof(TOut);
}
// TIn: operand element type (float -> tf32 MMA, bf16 -> f16-kind MMA); TOut: stored type.
// (kAMN, kBMN): operand majorness of problem 0; (kAMN1, kBMN1): that of problem 1 when kNP = 2.
// Each problem's majorness stays a compile-time constant: every role selects the problem of a
// work item with one warp-uniform branch and runs a loop instantiated for it.
template <typename TIn, typename TOut, bool kAMN, bool kBMN, int BN, int kCtas, int kNP = 1,
          bool kAMN1 = false, bool kBMN1 = false>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ GemmParams<TOut, kNP> P) {
  static_assert(kNP == 1 || kNP == 2, "one or two problems");
  pdl_launch_dependents();
  if (threadIdx.x == 0) {
    trace_mark(P.p[0].s, 0);
    trace_mark(P.p[0].s, 9, true);
  }
  using Tr = GemmTraits<TIn>;
  constexpr int BK = Tr::kBK;
  constexpr int kStages = gemm_stages<BN, kCtas>();
  constexpr int kTileM = kBM * kCtas;           // rows of the (pair's) output tile
  constexpr int kBNLocal = BN / kCtas;          // B rows (output columns) staged by this CTA
  constexpr int kABytes = kBM * kSwizzleBytes;  // 16 KiB
  constexpr int kBBytes = kBNLocal * kSwizzleBytes;
  constexpr int kChunk = kSwizzleBytes / sizeof(TIn);  // MN elements per 128-B swizzle row
  constexpr int kTmemCols = 2 * BN;                    // double-buffered fp32 accumulator
  static_assert(kTmemCols <= 512 && (kTmemCols & (kTmemCols - 1)) == 0, "TMEM cols");

  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - smem_u32(smem_raw));
  uint8_t* smA = smem;
  uint8_t* smB = smem + kStages * kABytes;
  uint8_t* smEpi = smem + kStages * (kABytes + kBBytes);  // 1 KiB aligned (stages are KiB multiples)
  uint8_t* smFeat = smEpi + kEpiStageBytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kStages * (kABytes + kBBytes) +
                                               kEpiStageBytes + kEpiFeatBytes);
  uint64_t* full_bar = bars;                    // [kStages]  (kCtas = 2: the leader's is used)
  uint64_t* empty_bar = bars + kStages;         // [kStages]
  uint64_t* tfull_bar = bars + 2 * kStages;     // [2]
  uint64_t* tempty_bar = bars + 2 * kStages + 2;  // [2]  (kCtas = 2: the leader's is used)
  uint64_t* feat_bar = bars + 2 * kStages + 4;    // [4 warps][kFeatBufs]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 4 + 4 * kFeatBufs);

  const int warp = uniform_warp_idx();  // provably warp-uniform: see the MMA issuer below
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = kCtas == 2 ? cluster_ctarank() : 0;
  const bool leader = cta_rank == 0;
  const int unit = blockIdx.x / kCtas;        // tile scheduler unit: a CTA or a CTA pair
  const int num_units = gridDim.x / kCtas;

  // Work item = (problem, split, tile): consecutive units take different tiles of the same K split.
  auto tiles_of = [](const GemmShape& s) {
    return ((s.M + kTileM - 1) / kTileM) * ((s.N + BN - 1) / BN) * s.batch;
  };
  int num_work = tiles_of(P.p[0].s) * P.p[0].s.splits;
  if constexpr (kNP == 2) num_work += tiles_of(P.p[1].s) * P.p[1].s.splits;
  // body(problem, item index within the problem, kAMN tag, kBMN tag) for flat work item `work`
  auto with_item = [&](int work, auto&& body) {
    if constexpr (kNP == 1) {
      body(P.p[0], work, std::bool_constant<kAMN>{}, std::bool_constant<kBMN>{});
    } else {
      const bool in_first = work < P.first_work;
      const int w = in_first ? work : work - P.first_work;
      if (in_first == (P.first == 0))
        body(P.p[0], w, std::bool_constant<kAMN>{}, std::bool_constant<kBMN>{});
      else
        body(P.p[1], w, std::bool_constant<kAMN1>{}, std::bool_constant<kBMN1>{});
    }
  };
  // the same for a body that does not depend on the operand majorness: one instance, problem
  // selected by a runtime index
  auto with_problem = [&](int work, auto&& body) {
    if constexpr (kNP == 1) {
      body(P.p[0], work);
    } else {
      const bool in_first = work < P.first_work;
      body(P.p[in_first ? P.first : 1 - P.first], in_first ? work : work - P.first_work);
    }
  };

  if (warp == 0 && lane == 0) {
#pragma unroll
    for (int i = 0; i < kNP; ++i) {
      tma_prefetch_desc(&P.p[i].tmapA);
      tma_prefetch_desc(&P.p[i].tmapB);
      if (P.p[i].s.tma_store) tma_prefetch_desc(&P.p[i].tmapC);
      if (P.p[i].s.feat_tma) tma_prefetch_desc(&P.p[i].tmapF);
    }
  }
  if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < kStages; ++i) {
        mbar_init(&full_bar[i], kCtas);  // one producer arrive per CTA of the pair
        mbar_init(&empty_bar[i], 1);
      }
      for (int i = 0; i < 2; ++i) {
        mbar_init(&tfull_bar[i], 1);
        mbar_init(&tempty_bar[i], 4 * kCtas);  // one arrive per epilogue warp (of both CTAs)
      }
      for (int i = 0; i < 4 * kFeatBufs; ++i) mbar_init(&feat_bar[i], 1);
      fence_mbar_init();
    }
    __syncwarp();
    if (kCtas == 2)
      tmem_alloc_2cta<kTmemCols>(tmem_slot);
    else
      tmem_alloc<kTmemCols>(tmem_slot);
  }
  tc_fence_before();
  if (kCtas == 2)
    cluster_sync_all();  // peer barriers must be initialised before any remote arrive / TMA credit
  else
    __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);  // warp-uniform value
  // Everything above overlapped the previous kernel's tail (programmatic dependent launch);
  // from here on this grid reads and writes global memory.
  if (threadIdx.x == 0) trace_mark(P.p[0].s, 1);
  pdl_wait();
  if (threadIdx.x == 0) trace_mark(P.p[0].s, 2);

  if (warp == 0) {
    // ===================== TMA producer (one per CTA) =====================
    if (lane == 0) {
      uint32_t stage = 0, phase = 0;
      for (int work = unit; work < num_work; work += num_units)
        with_item(work, [&](const GemmProblem<TOut>& pr, int item, auto amn, auto bmn) {
        constexpr bool kA = decltype(amn)::value, kB = decltype(bmn)::value;
        const GemmShape& s = pr.s;
        const int tiles_m = (s.M + kTileM - 1) / kTileM;
        const int tiles_per_batch = tiles_m * ((s.N + BN - 1) / BN);
        const int num_tiles = tiles_per_batch * s.batch;
        const int num_kb = (s.K + BK - 1) / BK;
        const int split = item / num_tiles;
        const int tile = item - split * num_tiles;
        const int b = tile / tiles_per_batch;
        const int t = tile - b * tiles_per_batch;
        const int m0 = (t % tiles_m) * kTileM + (int)cta_rank * kBM;
        const int n0 = (t / tiles_m) * BN + (int)cta_rank * kBNLocal;
        const int kb0 = split * s.kb_per_split;
        const int kb1 = min(kb0 + s.kb_per_split, num_kb);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1);
          if (kCtas == 1) {
            mbar_expect_tx(&full_bar[stage], kABytes + kBBytes);
          } else if (leader) {
            mbar_expect_tx(&full_bar[stage], 2 * (kABytes + kBBytes));  // both CTAs' bytes
          } else {
            mbar_arrive_remote(&full_bar[stage], 0);
          }
          int k0 = kb * BK;
          int cv_c0 = 0, cv_r = 0, cv_s = 0;
          if (s.conv_a && !kA) {  // kb -> (tap, channel block); B rows follow HWIO: (tap * C + c0)
            const int tap = kb / s.cv_cblocks;
            cv_c0 = (kb - tap * s.cv_cblocks) * BK;
            cv_r = tap / s.cv_S;
            cv_s = tap - cv_r * s.cv_S;
            k0 = tap * s.cv_C + cv_c0;
          }
          uint8_t* a_dst = smA + stage * kABytes;
          uint8_t* b_dst = smB + stage * kBBytes;
          auto load = [&](void* dst, const CUtensorMap* map, int c0, int c1) {
            if (kCtas == 2)
              tma_load_3d_2cta(dst, map, &full_bar[stage], c0, c1, b);
            else
              tma_load_3d(dst, map, &full_bar[stage], c0, c1, b);
          };
          // MN-major tile = [chunks][BK rows][128 B]; a 4-D map (128B, K, chunk, batch) fetches
          // all chunks with ONE instruction (TMA issue rate matters: 8 loads/stage cost ~30%).
          auto load4 = [&](void* dst, const CUtensorMap* map, int mn0) {
            if (kCtas == 2)
              tma_load_4d_2cta(dst, map, &full_bar[stage], 0, k0, mn0 / kChunk, b);
            else
              tma_load_4d(dst, map, &full_bar[stage], 0, k0, mn0 / kChunk, b);
          };
          if (!kA && s.conv_a) {
            // first output pixel of this CTA's 128-row slab -> input-space base coordinates
            const int ow = m0 % s.cv_OW;
            const int t2 = m0 / s.cv_OW;
            const int oh = t2 % s.cv_OH;
            const int img = t2 / s.cv_OH;
            const int bw = ow * s.cv_sw - s.cv_pl, bh = oh * s.cv_sh - s.cv_pt;
            if (kCtas == 2)
              tma_load_im2col_4d_2cta(a_dst, &pr.tmapA, &full_bar[stage], cv_c0, bw, bh, img,
                                      (uint16_t)cv_s, (uint16_t)cv_r);
            else
              tma_load_im2col_4d(a_dst, &pr.tmapA, &full_bar[stage], cv_c0, bw, bh, img,
                                 (uint16_t)cv_s, (uint16_t)cv_r);
          } else if (!kA) {
            load(a_dst, &pr.tmapA, k0, m0);
          } else if (s.conv_a) {
            // Filter gradient: GEMM-K runs over output pixels, GEMM-M over (tap, channel).  Each
            // 128-byte chunk of M is one (tap, channel block): an im2col box of BK pixels x chunk
            // channels lands in smem as [BK rows][128 B] -- the MN-major chunk layout.
            const int p0 = kb * BK;
            const int ow = p0 % s.cv_OW;
            const int t2 = p0 / s.cv_OW;
            const int oh = t2 % s.cv_OH;
            const int img = t2 / s.cv_OH;
            const int bw = ow * s.cv_sw - s.cv_pl, bh = oh * s.cv_sh - s.cv_pt;
#pragma unroll
            for (int c = 0; c < kBM / kChunk; ++c) {
              const int mi = m0 + c * kChunk;
              int tap = mi / s.cv_C;
              const int c0 = mi - tap * s.cv_C;
              if (tap >= s.cv_taps) tap = s.cv_taps - 1;  // rows beyond R*S*C are never stored
              const int fr = tap / s.cv_S, fs = tap - fr * s.cv_S;
              if (kCtas == 2)
                tma_load_im2col_4d_2cta(a_dst + c * (BK * kSwizzleBytes), &pr.tmapA, &full_bar[stage],
                                        c0, bw, bh, img, (uint16_t)fs, (uint16_t)fr);
              else
                tma_load_im2col_4d(a_dst + c * (BK * kSwizzleBytes), &pr.tmapA, &full_bar[stage], c0,
                                   bw, bh, img, (uint16_t)fs, (uint16_t)fr);
            }
          } else if (s.a_map4d) {
            load4(a_dst, &pr.tmapA, m0);
          } else {
#pragma unroll
            for (int c = 0; c < kBM / kChunk; ++c)
              load(a_dst + c * (BK * kSwizzleBytes), &pr.tmapA, m0 + c * kChunk, k0);
          }
          if (!kB) {
            load(b_dst, &pr.tmapB, k0, n0);
          } else if (s.b_map4d) {
            load4(b_dst, &pr.tmapB, n0);
          } else {
#pragma unroll
            for (int c = 0; c < kBNLocal / kChunk; ++c)
              load(b_dst + c * (BK * kSwizzleBytes), &pr.tmapB, n0 + c * kChunk, k0);
          }
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
      });
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (leader CTA only when paired) =====================
    // The WHOLE warp runs this loop and one elected lane issues each tcgen05 instruction
    // (predication inside the asm block).  Issuing from an `if (lane == 0)` region made ptxas
    // wrap every MMA in an ELECT + 5 x R2UR.BROADCAST waterfall loop: ~160 cycles of issue per
    // MMA against the MMA's own 128 -- the main loop ran at the issue rate (profiles/r02_notes.md).
    if (leader) {
      uint32_t stage = 0, phase = 0;
      uint32_t acc = 0, acc_phase = 0;
      for (int work = unit; work < num_work; work += num_units)
        with_item(work, [&](const GemmProblem<TOut>& pr, int item, auto amn, auto bmn) {
        constexpr bool kA = decltype(amn)::value, kB = decltype(bmn)::value;
        constexpr uint32_t kIdesc = make_idesc(Tr::kFormat, kA, kB, kTileM, BN);
        // MN-major tf32 must use the 32-byte-atom 128B swizzle: 4-row (512 B) K groups.
        constexpr bool kMn32 = sizeof(TIn) == 4;
        // descriptors of stage 0, k step 0: later ones differ only in the start-address field
        const uint64_t adesc0 = kA ? make_smem_desc_sw128(smem_u32(smA), BK * kSwizzleBytes,
                                                          kMn32 ? 512 : 1024, kMn32 ? 1 : 2)
                                   : make_smem_desc_sw128(smem_u32(smA), 16, 1024);
        const uint64_t bdesc0 = kB ? make_smem_desc_sw128(smem_u32(smB), BK * kSwizzleBytes,
                                                          kMn32 ? 512 : 1024, kMn32 ? 1 : 2)
                                   : make_smem_desc_sw128(smem_u32(smB), 16, 1024);
        const uint32_t a_hi = (uint32_t)(adesc0 >> 32), b_hi = (uint32_t)(bdesc0 >> 32);
        // K-major: advance 32 B inside the 128-B swizzle row; MN-major: advance kUmmaK rows.
        constexpr uint32_t kAStep = (kA ? Tr::kUmmaK * kSwizzleBytes : Tr::kUmmaK * (int)sizeof(TIn)) >> 4;
        constexpr uint32_t kBStep = (kB ? Tr::kUmmaK * kSwizzleBytes : Tr::kUmmaK * (int)sizeof(TIn)) >> 4;
        const GemmShape& s = pr.s;
        const int num_tiles = tiles_of(s);
        const int num_kb = (s.K + BK - 1) / BK;
        const int split = item / num_tiles;
        const int kb0 = split * s.kb_per_split;
        const int kb1 = min(kb0 + s.kb_per_split, num_kb);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1);
        __syncwarp();
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + acc * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          __syncwarp();
          tc_fence_after();
          if (lane == 0 && kb == kb0 && work == unit) trace_mark(s, 3);
          const uint32_t a_lo0 = (uint32_t)adesc0 + ((stage * kABytes) >> 4);
          const uint32_t b_lo0 = (uint32_t)bdesc0 + ((stage * kBBytes) >> 4);
#pragma unroll
          for (int k = 0; k < BK / Tr::kUmmaK; ++k) {
            const uint32_t accum = ((kb - kb0) | k) != 0;
            const uint32_t a_lo = a_lo0 + k * kAStep, b_lo = b_lo0 + k * kBStep;
            if (kCtas == 2) {
              if (sizeof(TIn) == 4)
                umma_tf32_elect_lohi_2cta(d_tmem, a_lo, a_hi, b_lo, b_hi, kIdesc, accum);
              else
                umma_f16_elect_lohi_2cta(d_tmem, a_lo, a_hi, b_lo, b_hi, kIdesc, accum);
            } else {
              if (sizeof(TIn) == 4)
                umma_tf32_elect_lohi(d_tmem, a_lo, a_hi, b_lo, b_hi, kIdesc, accum);
              else
                umma_f16_elect_lohi(d_tmem, a_lo, a_hi, b_lo, b_hi, kIdesc, accum);
            }
          }
          // frees the smem slot (in both CTAs) once these MMAs retire
          if (kCtas == 2)
            umma_commit_elect_2cta(&empty_bar[stage]);
          else
            umma_commit_elect(&empty_bar[stage]);
          if (++stage == kStages) {
            stage = 0;
            phase ^= 1;
          }
        }
        // accumulator ready for the epilogue warps (of both CTAs)
        if (lane == 0 && work == unit) trace_mark(s, 4);
        if (kCtas == 2)
          umma_commit_elect_2cta(&tfull_bar[acc]);
        else
          umma_commit_elect(&tfull_bar[acc]);
        if (++acc == 2) {
          acc = 0;
          acc_phase ^= 1;
        }
      });
    }
  } else {
    // ===================== epilogue warps =====================
    // TMEM -> registers (thread = output row) -> [bias / relu / relu-grad] -> 128B-swizzled smem
    // staging -> TMA store (coalesced, clips ragged edges).  Direct global stores remain as the
    // fallback for outputs TMA cannot address.
    constexpr int kEpiCols = kSwizzleBytes / (int)sizeof(TOut);  // columns per 128-B staged row
    constexpr int kLdPerIter = kEpiCols / 32;                    // tcgen05.ld x32 per iteration
    const int quad = warp & 3;  // TMEM lane quadrant this warp may access
    uint32_t acc = 0, acc_phase = 0;
    uint32_t ebuf = 0, stores_in_flight = 0;
    uint8_t* my_stage = smEpi + quad * 2 * kEpiBufBytes;
    uint8_t* my_feat = smFeat + quad * kFeatBufs * kEpiBufBytes;
    uint64_t* my_fbar = feat_bar + quad * kFeatBufs;
    uint32_t feat_issued = 0, feat_used = 0;  // running chunk counters (buffer = n % kFeatBufs)
    for (int work = unit; work < num_work; work += num_units)
      with_problem(work, [&](const GemmProblem<TOut>& pr, int item) {
      const GemmShape& s = pr.s;
      TOut* __restrict__ C = pr.C;
      const int tiles_m = (s.M + kTileM - 1) / kTileM;
      const int tiles_per_batch = tiles_m * ((s.N + BN - 1) / BN);
      const int num_tiles = tiles_per_batch * s.batch;
      const bool feat_on = s.relu_grad_features != nullptr && s.feat_tma && s.splits == 1;
      // ReluGrad features do not depend on the MMA: fetch them (coalesced, via TMA) ahead of use.
      auto issue_feat = [&](int col, int row0f, int bidx) {
        if (lane == 0) {
          uint64_t* fb = &my_fbar[feat_issued % kFeatBufs];
          mbar_expect_tx(fb, kEpiBufBytes);
          tma_load_3d(my_feat + (feat_issued % kFeatBufs) * kEpiBufBytes, &pr.tmapF, fb, col,
                      row0f, bidx);
        }
        ++feat_issued;
      };
      const bool vec_ok = (s.ldc % (16 / (int)sizeof(TOut)) == 0) &&
                          (s.strideC % (16 / (int)sizeof(TOut)) == 0) &&
                          ((reinterpret_cast<uintptr_t>(C) & 15) == 0);
      const int split = item / num_tiles;
      const int tile = item - split * num_tiles;
      const int b = tile / tiles_per_batch;
      const int t = tile - b * tiles_per_batch;
      const int m0 = (t % tiles_m) * kTileM + (int)cta_rank * kBM;
      const int n0 = (t / tiles_m) * BN;
      const int row0 = m0 + quad * 32;
      // the other problem's last item may have staged its bias here with generic stores
      if (kNP == 2 && feat_on && lane == 0) fence_proxy_async_smem();
      if (feat_on) {  // the first kFeatBufs chunks of this tile, while the MMAs are still running
#pragma unroll
        for (int pc = 0; pc < kFeatBufs; ++pc)
          if (pc * kEpiCols < BN && n0 + pc * kEpiCols < s.N) issue_feat(n0 + pc * kEpiCols, row0, b);
      }
      // Bias slice of this tile -> this warp's (otherwise unused) feature staging, also ahead of
      // the accumulator: the per-chunk broadcast reads then hit smem instead of exposing an L2
      // round trip per chunk.
      const bool bias_smem = s.bias != nullptr && s.bias_vec && s.splits == 1 && !feat_on &&
                             n0 + BN <= s.N;
      if (bias_smem) {
        const uint4* bsrc = reinterpret_cast<const uint4*>(static_cast<const TOut*>(s.bias) + n0);
        uint4* bdst = reinterpret_cast<uint4*>(my_feat);
        constexpr int kVecs = BN * (int)sizeof(TOut) / 16;
        for (int i = lane; i < kVecs; i += 32) bdst[i] = __ldg(bsrc + i);
        __syncwarp();
      }
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      if (work == unit && warp == 2 && lane == 0) trace_mark(s, 5);
      const int row = row0 + lane;
      const bool partial_out = s.splits > 1;
      TOut* crow = C + (long long)b * s.strideC + (long long)row * s.ldc;
      // split-K: fp32 partial tile, dense [split][batch][M][N]
      float* prow = s.partial + (((long long)split * s.batch + b) * s.M + row) * (long long)s.N;
      const bool pvec = (s.N & 3) == 0;
      const int cols_per_iter = partial_out ? 32 : kEpiCols;
      const int iters = BN / cols_per_iter;
#pragma unroll 1
      for (int c = 0; c < iters; ++c) {
        const int col = n0 + c * cols_per_iter;
        if (col >= s.N) break;  // warp-uniform
        uint32_t v[32 * kLdPerIter];
        {
          uint32_t(&v0)[32] = *reinterpret_cast<uint32_t(*)[32]>(&v[0]);
          tmem_ld_32x32(tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + c * cols_per_iter,
                        v0);
          if (kLdPerIter == 2 && !partial_out) {
            uint32_t(&v1)[32] = *reinterpret_cast<uint32_t(*)[32]>(&v[32 * (kLdPerIter - 1)]);
            tmem_ld_32x32(
                tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN + c * cols_per_iter + 32, v1);
          }
          tmem_ld_wait();
        }
        const int nvals = partial_out ? 32 : kEpiCols;
        // ---- fused element-wise tail (full-precision, before any rounding)
        if (!partial_out) {
          if (s.bias != nullptr) {
            const TOut* bp = static_cast<const TOut*>(s.bias) + col;
            if (s.bias_vec && col + kEpiCols <= s.N) {
              // every lane reads the same 128 bytes: 8 broadcast 16-byte loads
              const uint4* bsm = reinterpret_cast<const uint4*>(my_feat) + c * 8;
#pragma unroll
              for (int q4 = 0; q4 < 8; ++q4) {
                const uint4 bw = bias_smem ? bsm[q4] : __ldg(reinterpret_cast<const uint4*>(bp) + q4);
                const uint32_t bwv[4] = {bw.x, bw.y, bw.z, bw.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  if (sizeof(TOut) == 4) {
                    const int j = q4 * 4 + e;
                    v[j] = __float_as_uint(__uint_as_float(v[j]) + __uint_as_float(bwv[e]));
                  } else {
                    const int j = (q4 * 4 + e) * 2;
                    v[j % (32 * kLdPerIter)] = __float_as_uint(
                        __uint_as_float(v[j % (32 * kLdPerIter)]) + __uint_as_float(bwv[e] << 16));
                    v[(j + 1) % (32 * kLdPerIter)] =
                        __float_as_uint(__uint_as_float(v[(j + 1) % (32 * kLdPerIter)]) +
                                        __uint_as_float(bwv[e] & 0xFFFF0000u));
                  }
                }
              }
            } else {
#pragma unroll
              for (int j = 0; j < kEpiCols; ++j)
                if (col + j < s.N)
                  v[j] = __float_as_uint(__uint_as_float(v[j]) + ld_as_float(bp + j));
            }
          }
          if (s.relu) {
#pragma unroll
            for (int j = 0; j < kEpiCols; ++j) {
              const float f = __uint_as_float(v[j]);
              v[j] = __float_as_uint(f > 0.f ? f : 0.f);
            }
          }
          if (feat_on) {
            // this chunk's features were staged by TMA as [32 rows][128 B], 128B-swizzled
            mbar_wait(&my_fbar[feat_used % kFeatBufs], (feat_used / kFeatBufs) & 1);
            const uint32_t fbase =
                smem_u32(my_feat + (feat_used % kFeatBufs) * kEpiBufBytes) + lane * kSwizzleBytes;
#pragma unroll
            for (int q4 = 0; q4 < 8; ++q4) {
              uint32_t f0, f1, f2, f3;
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(f0), "=r"(f1), "=r"(f2), "=r"(f3)
                           : "r"(fbase + (uint32_t)((q4 ^ (lane & 7)) << 4)));
              const uint32_t fw[4] = {f0, f1, f2, f3};
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                if (sizeof(TOut) == 4) {
                  const int j = q4 * 4 + e;
                  const float g = __uint_as_float(v[j]);
                  v[j] = __float_as_uint(__uint_as_float(fw[e]) > 0.f ? g : g * 0.f);
                } else {
                  const int j0 = ((q4 * 4 + e) * 2) % (32 * kLdPerIter);
                  const int j1 = ((q4 * 4 + e) * 2 + 1) % (32 * kLdPerIter);
                  const float g0 = __uint_as_float(v[j0]), g1 = __uint_as_float(v[j1]);
                  v[j0] = __float_as_uint(__uint_as_float(fw[e] << 16) > 0.f ? g0 : g0 * 0.f);
                  v[j1] = __float_as_uint(__uint_as_float(fw[e] & 0xFFFF0000u) > 0.f ? g1
                                                                                      : g1 * 0.f);
                }
              }
            }
            ++feat_used;
            __syncwarp();  // every lane has read the buffer: it may be refilled
            const int next_col = col + kFeatBufs * kEpiCols;
            if (c + kFeatBufs < iters && next_col < s.N) issue_feat(next_col, row0, b);
          } else if (s.relu_grad_features != nullptr && row < s.M) {
            const TOut* fp = static_cast<const TOut*>(s.relu_grad_features) +
                             (long long)row * s.ld_features + col;
#pragma unroll
            for (int j = 0; j < kEpiCols; ++j)
              if (col + j < s.N) {
                const float g = __uint_as_float(v[j]);
                v[j] = __float_as_uint(ld_as_float(fp + j) > 0.f ? g : g * 0.f);
              }
          }
        }
        if (s.tma_store) {
          // pack to the output type: 32 x 32-bit words = one 128-byte staged row per thread
          uint32_t w[32];
          if (sizeof(TOut) == 4 || partial_out) {
#pragma unroll
            for (int j = 0; j < 32; ++j) w[j] = v[j];
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              __nv_bfloat162 h = __floats2bfloat162_rn(__uint_as_float(v[(2 * j) % nvals_max<TOut>()]),
                                                       __uint_as_float(v[(2 * j + 1) % nvals_max<TOut>()]));
              w[j] = *reinterpret_cast<uint32_t*>(&h);
            }
          }
          // the staging buffer we are about to overwrite must have been read by its TMA store
          if (stores_in_flight >= 2) {
            if (lane == 0) tma_store_wait_read<1>();
            __syncwarp();
          }
          uint8_t* buf = my_stage + ebuf * kEpiBufBytes;
          const uint32_t rbase = smem_u32(buf) + lane * kSwizzleBytes;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const uint32_t addr = rbase + (uint32_t)((j ^ (lane & 7)) << 4);  // 128B swizzle
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(w[4 * j]),
                         "r"(w[4 * j + 1]), "r"(w[4 * j + 2]), "r"(w[4 * j + 3])
                         : "memory");
          }
          fence_proxy_async_smem();
          __syncwarp();
          if (lane == 0) {
            tma_store_3d(&pr.tmapC, buf, col, row0, partial_out ? split * s.batch + b : b);
            tma_store_commit();
          }
          ++stores_in_flight;
          ebuf ^= 1;
        } else {
          int ncols = s.N - col;
          ncols = ncols > nvals ? nvals : ncols;
          if (row < s.M) {
            if (partial_out) {
              uint32_t(&v0)[32] = *reinterpret_cast<uint32_t(*)[32]>(&v[0]);
              store_row32(prow + col, v0, ncols, pvec);
            } else {
#pragma unroll
              for (int h = 0; h < kLdPerIter; ++h) {
                uint32_t(&vh)[32] = *reinterpret_cast<uint32_t(*)[32]>(&v[32 * h]);
                const int nc = ncols - 32 * h;
                if (nc > 0) store_row32(crow + col + 32 * h, vh, nc > 32 ? 32 : nc, vec_ok);
              }
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (kCtas == 2 && !leader)
          mbar_arrive_remote(&tempty_bar[acc], 0);  // the leader's MMA thread waits on it
        else
          mbar_arrive(&tempty_bar[acc]);
      }
      if (++acc == 2) {
        acc = 0;
        acc_phase ^= 1;
      }
    });
    if (warp == 2 && lane == 0) trace_mark(P.p[0].s, 6);
    if ((P.p[0].s.tma_store || P.p[kNP - 1].s.tma_store) && lane == 0)
      tma_store_wait<0>();  // global writes done before exit
    if (warp == 2 && lane == 0) trace_mark(P.p[0].s, 7);
  }

  tc_fence_before();
  if (kCtas == 2)
    cluster_sync_all();  // no CTA may exit (or free TMEM) while its peer can still signal it
  else
    __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    if (kCtas == 2)
      tmem_dealloc_2cta<kTmemCols>(tmem_base);
    else
      tmem_dealloc<kTmemCols>(tmem_base);
  }
  if (threadIdx.x == 0) {
    trace_mark(P.p[0].s, 8);
    trace_mark(P.p[0].s, 10, true);
  }
}

// Split-K reduction: out = sum over splits (ascending, deterministic) of the fp32 partials.
template <typename TOut>
__global__ void __launch_bounds__(256)
splitk_reduce_kernel(const float* __restrict__ partial, TOut* __restrict__ C, int splits,
                     long long batch, int M, int N, int ldc, long long strideC,
                     const TOut* __restrict__ bias, int relu) {
  pdl_launch_dependents();
  pdl_wait();  // launched programmatically behind the GEMM that writes `partial`
  const long long per_split = batch * (long long)M * N;
  const int n4 = (N + 3) / 4;
  const long long total = batch * (long long)M * n4;
  // persistent grid-stride over 4-column groups
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total;
       i += (long long)gridDim.x * 256) {
  const int c4 = (int)(i % n4);
  const long long r = i / n4;  // b * M + row
  const long long b = r / M;
  const int row = (int)(r - b * M);
  const int col = c4 * 4;
  const int nc = min(4, N - col);
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  const float* p = partial + r * N + col;
  for (int s = 0; s < splits; ++s) {
    if (nc == 4 && (N & 3) == 0) {
      const float4 v = *reinterpret_cast<const float4*>(p + s * per_split);
      acc[0] += v.x;
      acc[1] += v.y;
      acc[2] += v.z;
      acc[3] += v.w;
    } else {
      for (int j = 0; j < nc; ++j) acc[j] += p[s * per_split + j];
    }
  }
  TOut* dst = C + b * strideC + (long long)row * ldc + col;
  if (bias != nullptr) {  // fused tail of a split GEMM: + bias[col], then relu (full-precision sum)
    for (int j = 0; j < nc; ++j) {
      acc[j] += ld_as_float(bias + col + j);
      if (relu) acc[j] = acc[j] > 0.f ? acc[j] : 0.f;
    }
  }
  for (int j = 0; j < nc; ++j) {
    if (sizeof(TOut) == 4)
      reinterpret_cast<float*>(dst)[j] = acc[j];
    else
      reinterpret_cast<__nv_bfloat16*>(dst)[j] = __float2bfloat16_rn(acc[j]);
  }
  }  // group loop
}

// Contiguous fast path (C is [batch * M, N] with ldc == N, N % 4 == 0): one 16-byte column group per
// thread and no index arithmetic beyond the bias column.  All S partial loads are issued before the
// first add (S is a template parameter, so they sit in registers); the adds keep the ascending
// split order of the generic kernel, i.e. the result is bit-identical.
template <typename TOut, int S>
__global__ void __launch_bounds__(256)
splitk_reduce_flat_kernel(const float4* __restrict__ partial, TOut* __restrict__ C,
                          long long per_split4, long long total4, int n4,
                          const TOut* __restrict__ bias, int relu) {
  pdl_launch_dependents();
  pdl_wait();
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total4;
       i += (long long)gridDim.x * 256) {
    float4 v[S];
#pragma unroll
    for (int s = 0; s < S; ++s) v[s] = __ldcg(partial + i + s * per_split4);
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int s = 0; s < S; ++s) {
      acc[0] += v[s].x;
      acc[1] += v[s].y;
      acc[2] += v[s].z;
      acc[3] += v[s].w;
    }
    if (bias != nullptr) {
      const int col = (int)(i % n4) * 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        acc[j] += ld_as_float(bias + col + j);
        if (relu) acc[j] = acc[j] > 0.f ? acc[j] : 0.f;
      }
    }
    if (sizeof(TOut) == 4) {
      reinterpret_cast<float4*>(C)[i] = make_float4(acc[0], acc[1], acc[2], acc[3]);
    } else {
      const __nv_bfloat162 lo = __floats2bfloat162_rn(acc[0], acc[1]);
      const __nv_bfloat162 hi = __floats2bfloat162_rn(acc[2], acc[3]);
      reinterpret_cast<uint2*>(C)[i] = make_uint2(*reinterpret_cast<const uint32_t*>(&lo),
                                                  *reinterpret_cast<const uint32_t*>(&hi));
    }
  }
}

// ------------------------------------------------------------------ host side

// Operand description: row-major matrix [rows, cols] per batch, leading dimension ld (elements).
//   K-major  operand: rows = MN extent, cols = K.
//   MN-major operand: rows = K,         cols = MN extent.
static int encode_operand_map(CUtensorMap* map, CUtensorMapDataType dt, size_t esize,
                              const void* ptr, long long rows, long long cols, long long ld,
                              long long batch, long long batch_stride, int box_inner,
                              int box_rows, bool mn_major) {
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batch};
  cuuint64_t gstride[2] = {(cuuint64_t)(ld * esize),
                           (cuuint64_t)((batch > 1 ? batch_stride : rows * ld) * esize)};
  cuuint32_t box[3] = {(cuuint32_t)box_inner, (cuuint32_t)box_rows, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = driver().cuTensorMapEncodeTiled(
      map, dt, 3, const_cast<void*>(ptr), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
      // MN-major fp32 (tf32) tiles need 32-byte swizzle atoms (UMMA SWIZZLE_128B_BASE32B)
      (mn_major && esize == 4) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
      CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)",
                   (int)r, rows, cols, ld);
    return B200_INTERNAL;
  }
  return B200_OK;
}

// MN-major operand stored [K, MN] (ld elements per row), MN % chunk == 0: 4-D view
// (chunk, K, MN / chunk, batch) so that one box {chunk, BK, nchunks, 1} lands in smem as
// [nchunks][BK][128 B] -- the UMMA MN-major tile layout.
static bool encode_mn_major_map4d(CUtensorMap* map, CUtensorMapDataType dt, size_t esize,
                                  const void* ptr, long long K, long long MN, long long ld,
                                  long long batch, long long batch_stride, int chunk, int bk,
                                  int nchunks) {
  if (MN % chunk != 0) return false;
  cuuint64_t gdim[4] = {(cuuint64_t)chunk, (cuuint64_t)K, (cuuint64_t)(MN / chunk),
                        (cuuint64_t)batch};
  cuuint64_t gstride[3] = {(cuuint64_t)(ld * esize), (cuuint64_t)(chunk * esize),
                           (cuuint64_t)((batch > 1 ? batch_stride : K * ld) * esize)};
  cuuint32_t box[4] = {(cuuint32_t)chunk, (cuuint32_t)bk, (cuuint32_t)nchunks, 1};
  cuuint32_t estr[4] = {1, 1, 1, 1};
  return driver().cuTensorMapEncodeTiled(
             map, dt, 4, const_cast<void*>(ptr), gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE,
             esize == 4 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

bool conv_a_supported(int dtype, const ConvAOperand& c) {
  const int es = dtype == B200_DT_FLOAT ? 4 : 2;
  const int bk = kSwizzleBytes / es;
  if (!driver().cuTensorMapEncodeIm2col) return false;
  if (c.C % bk != 0) return false;                      // whole 128-byte channel blocks per tap
  if ((reinterpret_cast<uintptr_t>(c.input) & 15) != 0) return false;
  const int pad_r = std::max(0, (c.OW - 1) * c.sw + c.S - c.W) - c.pl;
  const int pad_b = std::max(0, (c.OH - 1) * c.sh + c.R - c.H) - c.pt;
  const int lo_w = -c.pl, lo_h = -c.pt, up_w = pad_r - (c.S - 1), up_h = pad_b - (c.R - 1);
  for (int v : {lo_w, lo_h, up_w, up_h})
    if (v < -128 || v > 127) return false;              // rank-4 corner range
  if (c.S > 256 || c.R > 256 || c.sw > 8 || c.sh > 8) return false;
  if ((long long)c.N * c.OH * c.OW > 0x7fffffffLL) return false;
  return true;
}

static int encode_im2col_map(CUtensorMap* map, CUtensorMapDataType dt, size_t esize,
                             const ConvAOperand& c, int channels_per_pixel, int pixels,
                             bool mn_major = false) {
  cuuint64_t gdim[4] = {(cuuint64_t)c.C, (cuuint64_t)c.W, (cuuint64_t)c.H, (cuuint64_t)c.N};
  cuuint64_t gstride[3] = {(cuuint64_t)c.C * esize, (cuuint64_t)c.W * c.C * esize,
                           (cuuint64_t)c.H * c.W * c.C * esize};
  const int pad_r = std::max(0, (c.OW - 1) * c.sw + c.S - c.W) - c.pl;
  const int pad_b = std::max(0, (c.OH - 1) * c.sh + c.R - c.H) - c.pt;
  int lower[2] = {-c.pl, -c.pt};                         // {W, H}
  int upper[2] = {pad_r - (c.S - 1), pad_b - (c.R - 1)};
  cuuint32_t estr[4] = {1, (cuuint32_t)c.sw, (cuuint32_t)c.sh, 1};
  CUresult r = driver().cuTensorMapEncodeIm2col(
      map, dt, 4, const_cast<void*>(c.input), gdim, gstride, lower, upper,
      (cuuint32_t)channels_per_pixel, (cuuint32_t)pixels, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
      (mn_major && esize == 4) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
      CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_last_error("cuTensorMapEncodeIm2col failed with CUresult %d", (int)r);
    return B200_INTERNAL;
  }
  return B200_OK;
}

// Output (or split-K partial) tensor map for the epilogue's TMA stores: box = 128 B x 32 rows.
static bool encode_store_map(CUtensorMap* map, CUtensorMapDataType dt, size_t esize, void* ptr,
                             long long rows, long long cols, long long ld, long long batches,
                             long long batch_stride) {
  if ((ld * esize) % 16 || (batch_stride * esize) % 16 || (reinterpret_cast<uintptr_t>(ptr) & 15))
    return false;
  cuuint64_t gdim[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)batches};
  cuuint64_t gstride[2] = {(cuuint64_t)(ld * esize),
                           (cuuint64_t)((batches > 1 ? batch_stride : rows * ld) * esize)};
  cuuint32_t box[3] = {(cuuint32_t)(kSwizzleBytes / esize), 32, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  return driver().cuTensorMapEncodeTiled(map, dt, 3, ptr, gdim, gstride, box, estr,
                                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                         CU_TENSOR_MAP_L2_PROMOTION_NONE,
                                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Tensor maps and shape of one GEMM for a launch with BN x kCtas tiles.  The split-K plan is the
// one the GEMM's own launch uses, whether it runs alone or as one problem of a pair launch.
template <typename TIn, typename TOut, bool kAMN, bool kBMN, int BN, int kCtas>
static int prepare_problem(const GemmArgs& g, GemmProblem<TOut>& pr, long long* tiles_out) {
  using Tr = GemmTraits<TIn>;
  constexpr int kChunk = kSwizzleBytes / sizeof(TIn);
  constexpr int kTileM = kBM * kCtas;
  constexpr int kBNLocal = BN / kCtas;
  CUtensorMap& ma = pr.tmapA;
  CUtensorMap& mb = pr.tmapB;
  int rc;
  // A: logical [M,K]; stored [M,K] (K-major) or [K,M] (MN-major).  Box = one CTA's 128 rows.
  bool a4 = false, b4 = false;
  if (g.conv_a) {
    if (kAMN)  // filter gradient: boxes of BK pixels x one 128-byte channel chunk
      rc = encode_im2col_map(&ma, Tr::kTmaType, sizeof(TIn), *g.conv_a, kChunk, Tr::kBK, true);
    else       // forward / input gradient: boxes of 128 pixels x BK channels
      rc = encode_im2col_map(&ma, Tr::kTmaType, sizeof(TIn), *g.conv_a, Tr::kBK, kBM);
  } else if (!kAMN)
    rc = encode_operand_map(&ma, Tr::kTmaType, sizeof(TIn), g.a, g.M, g.K, g.lda, g.batch,
                            g.strideA, Tr::kBK, kBM, false);
  else if ((a4 = encode_mn_major_map4d(&ma, Tr::kTmaType, sizeof(TIn), g.a, g.K, g.M, g.lda,
                                       g.batch, g.strideA, kChunk, Tr::kBK, kBM / kChunk)))
    rc = B200_OK;
  else
    rc = encode_operand_map(&ma, Tr::kTmaType, sizeof(TIn), g.a, g.K, g.M, g.lda, g.batch,
                            g.strideA, kChunk, Tr::kBK, true);
  if (rc) return rc;
  // B: logical [K,N]; stored [K,N] (MN-major) or [N,K] (K-major).  Box = one CTA's BN/kCtas cols.
  if (!kBMN)
    rc = encode_operand_map(&mb, Tr::kTmaType, sizeof(TIn), g.b, g.N, g.K, g.ldb, g.batch,
                            g.strideB, Tr::kBK, kBNLocal, false);
  else if ((b4 = encode_mn_major_map4d(&mb, Tr::kTmaType, sizeof(TIn), g.b, g.K, g.N, g.ldb,
                                       g.batch, g.strideB, kChunk, Tr::kBK, kBNLocal / kChunk)))
    rc = B200_OK;
  else
    rc = encode_operand_map(&mb, Tr::kTmaType, sizeof(TIn), g.b, g.K, g.N, g.ldb, g.batch,
                            g.strideB, kChunk, Tr::kBK, true);
  if (rc) return rc;

  GemmShape& s = pr.s;
  memset(&s, 0, sizeof(s));
  pr.C = static_cast<TOut*>(g.c);
  s.M = (int)g.M;
  s.N = (int)g.N;
  s.K = (int)g.K;
  s.batch = (int)g.batch;
  s.ldc = (int)g.ldc;
  s.strideC = g.strideC;
  const long long tiles = ((g.M + kTileM - 1) / kTileM) * ((g.N + BN - 1) / BN) * g.batch;
  *tiles_out = tiles;
  const int units = sm_count() / kCtas;  // schedulable CTAs or CTA pairs
  // split-K when the output tiles alone cannot fill the SMs and scratch was provided
  const int num_kb = (int)((g.K + Tr::kBK - 1) / Tr::kBK);
  int splits = 1;
  // A ReluGrad tail needs the complete sum in the GEMM's own epilogue; a bias (+ relu) tail can
  // ride on the ordered reduction pass of a split GEMM (LeNet fc1: 512 x 1024 x 3136 has 8 pair
  // tiles for 74 pairs -- 43 us unsplit).
  const bool fused = g.relu_grad_features != nullptr;
  if (g.workspace && !fused) {
    splits = plan_splits(tiles, num_kb, units);
    while (splits > 1 &&
           (size_t)splits * g.batch * g.M * g.N * sizeof(float) > g.workspace_bytes)
      --splits;
    if (splits < 1) splits = 1;
  }
  s.kb_per_split = (num_kb + splits - 1) / splits;
  splits = (num_kb + s.kb_per_split - 1) / s.kb_per_split;  // no empty split
  s.splits = splits;
  s.partial = static_cast<float*>(g.workspace);
  s.a_map4d = a4 ? 1 : 0;
  s.conv_a = g.conv_a ? 1 : 0;
  if (g.conv_a) {
    const ConvAOperand& c = *g.conv_a;
    s.cv_OW = c.OW; s.cv_OH = c.OH; s.cv_sh = c.sh; s.cv_sw = c.sw; s.cv_pt = c.pt; s.cv_pl = c.pl;
    s.cv_S = c.S; s.cv_C = c.C; s.cv_cblocks = c.C / Tr::kBK; s.cv_taps = c.R * c.S;
  }
  s.b_map4d = b4 ? 1 : 0;
  s.bias = g.bias;
  s.relu = g.relu ? 1 : 0;
  s.relu_grad_features = g.relu_grad_features;
  s.ld_features = (int)g.ld_features;
  CUtensorMap& mc = pr.tmapC;
  memset(&mc, 0, sizeof(mc));
  if (splits > 1)
    s.tma_store = encode_store_map(&mc, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, g.workspace, g.M, g.N,
                                   g.N, (long long)splits * g.batch, g.M * g.N);
  else
    s.tma_store = encode_store_map(&mc, sizeof(TOut) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                                          : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                                   sizeof(TOut), g.c, g.M, g.N, g.ldc, g.batch, g.strideC);
  CUtensorMap& mf = pr.tmapF;
  memset(&mf, 0, sizeof(mf));
  s.feat_tma = 0;
  if (g.relu_grad_features && splits == 1)
    s.feat_tma = encode_store_map(&mf, sizeof(TOut) == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                                          : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16,
                                  sizeof(TOut), const_cast<void*>(g.relu_grad_features), g.M, g.N,
                                  g.ld_features, 1, g.M * g.ld_features);
  s.bias_vec = g.bias && (reinterpret_cast<uintptr_t>(g.bias) & 15) == 0;
  s.trace = nullptr;
  return B200_OK;
}

// Ordered reduction of a split GEMM's fp32 partials into C (+ its bias / relu tail).
template <typename TOut>
static int launch_splitk_reduce(const GemmArgs& g, const GemmShape& s, bool pdl, bool prof,
                                cudaStream_t stream) {
  const int splits = s.splits;
  const long long groups = g.batch * g.M * ((g.N + 3) / 4);
  long long rblocks = (groups + 255) / 256;
  if (rblocks > 8LL * sm_count()) rblocks = 8LL * sm_count();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)rblocks);
  cfg.blockDim = dim3(256);
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl && !prof ? 1 : 0;
  const bool flat = (s.N & 3) == 0 && s.ldc == s.N &&
                    (g.batch == 1 || (long long)s.strideC == (long long)s.M * s.N) &&
                    splits >= 2 && splits <= 16 &&
                    (reinterpret_cast<uintptr_t>(s.partial) & 15) == 0 &&
                    (reinterpret_cast<uintptr_t>(g.c) & 15) == 0;
  cudaError_t e;
  void* ktok = kernel_times_enabled() ? kernel_times_begin(stream) : nullptr;
  if (ktok) cfg.numAttrs = 0;
  if (flat) {
    const long long total4 = g.batch * (long long)s.M * (s.N / 4);
    const float4* p4 = reinterpret_cast<const float4*>(s.partial);
    TOut* c = static_cast<TOut*>(g.c);
    const TOut* bias = static_cast<const TOut*>(g.bias);
    const int relu = g.relu ? 1 : 0, n4 = s.N / 4;
    switch (splits) {
#define B200_SPLITK_FLAT(S_)                                                                   \
  case S_:                                                                                     \
    e = cudaLaunchKernelEx(&cfg, splitk_reduce_flat_kernel<TOut, S_>, p4, c, total4, total4, \
                           n4, bias, relu);                                                    \
    break;
      B200_SPLITK_FLAT(2)
      B200_SPLITK_FLAT(3)
      B200_SPLITK_FLAT(4)
      B200_SPLITK_FLAT(5)
      B200_SPLITK_FLAT(6)
      B200_SPLITK_FLAT(7)
      B200_SPLITK_FLAT(8)
      B200_SPLITK_FLAT(9)
      B200_SPLITK_FLAT(10)
      B200_SPLITK_FLAT(11)
      B200_SPLITK_FLAT(12)
      B200_SPLITK_FLAT(13)
      B200_SPLITK_FLAT(14)
      B200_SPLITK_FLAT(15)
      default:
      B200_SPLITK_FLAT(16)
#undef B200_SPLITK_FLAT
    }
  } else {
    e = cudaLaunchKernelEx(&cfg, splitk_reduce_kernel<TOut>,
                           static_cast<const float*>(s.partial), static_cast<TOut*>(g.c),
                           splits, (long long)g.batch, s.M, s.N, s.ldc,
                           (long long)s.strideC, static_cast<const TOut*>(g.bias),
                           g.relu ? 1 : 0);
  }
  if (ktok)
    kernel_times_end(ktok, stream,
                     flat ? reinterpret_cast<const void*>(splitk_reduce_flat_kernel<TOut, 4>)
                          : reinterpret_cast<const void*>(splitk_reduce_kernel<TOut>));
  if (e != cudaSuccess) {
    set_last_error("splitk_reduce launch: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return B200_INTERNAL;
  }
  note_launch();
  return B200_OK;
}

// One persistent launch over kNP problems, then one ordered reduction pass per split problem.
// kNP = 1: one GEMM.  kNP = 2: a dense layer's input gradient dX = dY * W^T (slot 0: both operands
// K-major) and weight gradient dW = X^T * dY (slot 1: both MN-major) with BN-wide pair tiles.  Each
// problem keeps the split plan, tile order and fused tail of its own launch, so every output is
// bit-identical to it; the problem whose items are longer comes first in the work list, so that
// the short items fill the tail.  The pair counts as one GEMM launch with the summed FLOPs.
template <typename TIn, typename TOut, bool kAMN, bool kBMN, int BN, int kCtas, int kNP = 1,
          bool kAMN1 = false, bool kBMN1 = false>
static int launch_gemm(const GemmArgs* const (&g)[kNP], cudaStream_t stream) {
  constexpr auto kern = gemm_tcgen05_kernel<TIn, TOut, kAMN, kBMN, BN, kCtas, kNP, kAMN1, kBMN1>;
  constexpr size_t smem = gemm_smem_bytes<BN, kCtas>();
  GemmParams<TOut, kNP> P;
  memset(&P, 0, sizeof(P));
  long long work[kNP], total_work = 0;
  double flops = 0.0;
  for (int i = 0; i < kNP; ++i) {
    long long tiles = 0;
    const int rc = i == 0 ? prepare_problem<TIn, TOut, kAMN, kBMN, BN, kCtas>(*g[0], P.p[0], &tiles)
                          : prepare_problem<TIn, TOut, kAMN1, kBMN1, BN, kCtas>(*g[i], P.p[i], &tiles);
    if (rc) return rc;
    work[i] = tiles * P.p[i].s.splits;
    total_work += work[i];
    flops += 2.0 * (double)g[i]->M * (double)g[i]->N * (double)g[i]->K * g[i]->batch;
  }
  if constexpr (kNP == 2) {
    P.first = P.p[1].s.kb_per_split > P.p[0].s.kb_per_split ? 1 : 0;
    P.first_work = (int)work[P.first];
  }
  static const bool trace_on = getenv("B200TF_GEMM_TRACE") != nullptr;
  static unsigned long long* trace_buf = nullptr;
  if (trace_on) {
    if (trace_buf == nullptr) cudaMalloc(&trace_buf, 16 * sizeof(unsigned long long));
    if (trace_buf != nullptr) {
      cudaMemsetAsync(trace_buf, 0, 16 * sizeof(unsigned long long), stream);
      cudaStreamSynchronize(stream);
      for (int i = 0; i < kNP; ++i) P.p[i].s.trace = trace_buf;
    }
  }
  static bool attr_set = false;  // per template instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)smem);
    if (e != cudaSuccess) {
      set_last_error("cudaFuncSetAttribute(smem=%zu): %s", smem, cudaGetErrorString(e));
      return B200_INTERNAL;
    }
    attr_set = true;
  }
  const bool prof = profile_enabled();
  const bool pdl = pdl_enabled();
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)std::min<long long>(total_work, sm_count() / kCtas) * kCtas);
  cfg.blockDim = dim3(kGemmThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[2];
  int na = 0;
  if (kCtas > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = kCtas;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
  }
  if (pdl) {  // prologue overlaps the predecessor's tail; the kernel pdl_wait()s before global I/O
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  cfg.attrs = attr;
  cfg.numAttrs = na;
  if (prof) profile_gemm_launch_begin(stream);
  void* ktok = kernel_times_enabled() ? kernel_times_begin(stream) : nullptr;
  cudaError_t e = cudaLaunchKernelEx(&cfg, kern, P);
  if (ktok) kernel_times_end(ktok, stream, reinterpret_cast<const void*>(kern));
  if (e != cudaSuccess) {
    set_last_error("gemm_tcgen05 launch: %s", cudaGetErrorString(e));
    cudaGetLastError();
    return B200_INTERNAL;
  }
  if (prof) profile_gemm_launch_end(stream, flops);
  if (P.p[0].s.trace != nullptr) {  // debug: phase boundaries, ns since the first CTA entered
    unsigned long long t[16];
    cudaStreamSynchronize(stream);
    cudaMemcpy(t, P.p[0].s.trace, sizeof(t), cudaMemcpyDeviceToHost);
    fprintf(stderr,
            "[gemm trace] %lldx%lldx%lld BN=%d ctas=%d problems=%d splits=%d: prologue %llu | "
            "pdl_wait %llu | first operands %llu | mainloop issued %llu | accumulator ready %llu | "
            "epilogue stored %llu | stores drained %llu | exit %llu | last CTA entry %lld exit "
            "%lld (ns since entry)\n",
            g[0]->M, g[0]->N, g[0]->K, BN, kCtas, kNP, P.p[0].s.splits, t[1] - t[0], t[2] - t[0],
            t[3] - t[0], t[4] - t[0], t[5] - t[0], t[6] - t[0], t[7] - t[0], t[8] - t[0],
            (long long)(t[9] - t[0]), (long long)(t[10] - t[0]));
  }
  note_launch();
  for (int i = 0; i < kNP; ++i)
    if (P.p[i].s.splits > 1) {
      const int rc = launch_splitk_reduce<TOut>(*g[i], P.p[i].s, pdl, prof, stream);
      if (rc) return rc;
    }
  return check_launch("gemm_tcgen05");
}

template <typename TIn, typename TOut, int BN, int kCtas>
static int dispatch_major(const GemmArgs& g, cudaStream_t stream) {
  const GemmArgs* const gs[1] = {&g};
  if (!g.a_mn_major && !g.b_mn_major)
    return launch_gemm<TIn, TOut, false, false, BN, kCtas>(gs, stream);
  if (!g.a_mn_major && g.b_mn_major)
    return launch_gemm<TIn, TOut, false, true, BN, kCtas>(gs, stream);
  if (g.a_mn_major && !g.b_mn_major)
    return launch_gemm<TIn, TOut, true, false, BN, kCtas>(gs, stream);
  return launch_gemm<TIn, TOut, true, true, BN, kCtas>(gs, stream);
}

// Split-K plan shared by the launcher and gemm_workspace_bytes(): how many K splits a tiling
// with `tiles` output tiles would use on `units` schedulable CTAs / CTA pairs (1 = none).
static int plan_splits(long long tiles, int num_kb, int units) {
  if (tiles * 2 > units || num_kb < 8) return 1;
  long long splits = units / tiles;
  if (splits > num_kb / 4) splits = num_kb / 4;  // >= 4 K blocks per split
  if (splits > 64) splits = 64;  // scratch = splits * M * N * 4 bytes; callers size it from this plan
  return splits < 1 ? 1 : (int)splits;
}

// Tile configuration.  CTA pairs (256 x BN tiles, cta_group::2) whenever the problem has at least
// one full pair tile of rows: they halve the L2->smem operand traffic per FLOP, which is what
// bounds the main loop.  Otherwise single CTAs with 128 x {128, 64} tiles.
struct TileConfig {
  int ctas, bn;
};
static TileConfig choose_config(const GemmArgs& g) {
  if (g.M >= 256 && g.N >= 128) return {2, g.N >= 256 ? 256 : 128};
  if (g.N <= 64) return {1, 64};
  const long long t128 = ((g.M + kBM - 1) / kBM) * ((g.N + 127) / 128) * g.batch;
  if (t128 >= sm_count()) return {1, 128};
  const int bk = g.dtype == B200_DT_FLOAT ? GemmTraits<float>::kBK : GemmTraits<__nv_bfloat16>::kBK;
  if (g.workspace && plan_splits(t128, (int)((g.K + bk - 1) / bk), sm_count()) > 1) return {1, 128};
  return {1, 64};
}

size_t gemm_workspace_bytes(int dtype, long long M, long long N, long long K, long long batch) {
  if (M <= 0 || N <= 0 || K <= 0 || batch <= 0) return 0;
  GemmArgs g{};
  g.dtype = dtype;
  g.M = M;
  g.N = N;
  g.K = K;
  g.batch = batch;
  g.workspace = reinterpret_cast<void*>(1);  // "scratch will be available"
  const TileConfig c = choose_config(g);
  const int bk = dtype == B200_DT_FLOAT ? GemmTraits<float>::kBK : GemmTraits<__nv_bfloat16>::kBK;
  const long long tiles = ((M + kBM * c.ctas - 1) / (kBM * c.ctas)) * ((N + c.bn - 1) / c.bn) * batch;
  const int splits = plan_splits(tiles, (int)((K + bk - 1) / bk), sm_count() / c.ctas);
  return splits > 1 ? (size_t)splits * batch * M * N * sizeof(float) : 0;
}

bool gemm_tcgen05_supported(const GemmArgs& g) {
  const int e = g.dtype == B200_DT_FLOAT ? 4 : 2;
  const int align = 16 / e;
  if (g.M <= 0 || g.N <= 0 || g.K <= 0 || g.batch <= 0) return false;
  if (g.conv_a) {
    if (g.ldb % align || (reinterpret_cast<uintptr_t>(g.b) & 15)) return false;
    return g.batch == 1 && conv_a_supported(g.dtype, *g.conv_a);
  }
  if (g.lda % align || g.ldb % align) return false;
  if (g.batch > 1 && (g.strideA % align || g.strideB % align)) return false;
  if ((reinterpret_cast<uintptr_t>(g.a) & 15) || (reinterpret_cast<uintptr_t>(g.b) & 15))
    return false;
  if (g.M > 0x7fffffffLL || g.N > 0x7fffffffLL || g.K > 0x7fffffffLL) return false;
  return true;
}

template <typename TIn, typename TOut>
static int dispatch_config(const GemmArgs& g, const TileConfig& c, cudaStream_t stream) {
  if (c.ctas == 2) {
    if (c.bn == 256) return dispatch_major<TIn, TOut, 256, 2>(g, stream);
    return dispatch_major<TIn, TOut, 128, 2>(g, stream);
  }
  if (c.bn == 64) return dispatch_major<TIn, TOut, 64, 1>(g, stream);
  return dispatch_major<TIn, TOut, 128, 1>(g, stream);
}

int gemm_tcgen05(const GemmArgs& g, cudaStream_t stream) {
  const TileConfig c = choose_config(g);
  if (g.dtype == B200_DT_FLOAT) return dispatch_config<float, float>(g, c, stream);
  if (g.dtype == B200_DT_BFLOAT16)
    return dispatch_config<__nv_bfloat16, __nv_bfloat16>(g, c, stream);
  set_last_error("gemm_tcgen05: unsupported dtype %d", g.dtype);
  return B200_UNIMPLEMENTED;
}

int gemm_tcgen05_pair(const GemmArgs& a, const GemmArgs& b, cudaStream_t stream) {
  auto majors = [](const GemmArgs& g, bool mn) { return g.a_mn_major == mn && g.b_mn_major == mn; };
  // slot 0 takes the K-major x K-major product, slot 1 the MN-major x MN-major one
  const bool a_first = majors(a, false) && majors(b, true);
  const GemmArgs& g0 = a_first ? a : b;
  const GemmArgs& g1 = a_first ? b : a;
  const TileConfig c0 = choose_config(g0), c1 = choose_config(g1);
  const bool paired = a.dtype == b.dtype && majors(g0, false) && majors(g1, true) &&
                      a.batch == 1 && b.batch == 1 && !a.conv_a && !b.conv_a &&
                      gemm_tcgen05_supported(a) && gemm_tcgen05_supported(b) && c0.ctas == 2 &&
                      c1.ctas == 2 && c0.bn == c1.bn;
  if (!paired) {
    const int rc = gemm_tcgen05(a, stream);
    return rc ? rc : gemm_tcgen05(b, stream);
  }
  const GemmArgs* const gs[2] = {&g0, &g1};
  using bf16 = __nv_bfloat16;
  if (g0.dtype == B200_DT_FLOAT)
    return c0.bn == 256 ? launch_gemm<float, float, false, false, 256, 2, 2, true, true>(gs, stream)
                        : launch_gemm<float, float, false, false, 128, 2, 2, true, true>(gs, stream);
  return c0.bn == 256 ? launch_gemm<bf16, bf16, false, false, 256, 2, 2, true, true>(gs, stream)
                      : launch_gemm<bf16, bf16, false, false, 128, 2, 2, true, true>(gs, stream);
}

}  // namespace b200
