// Reduction-style HBM-bound op kernels: BiasAddGrad, Softmax / LogSoftmax,
// SoftmaxCrossEntropyWithLogits, ArgMax, and a deterministic sum (loss glue).
//
// Reference kernels replaced (relative to tensorflow/core/kernels/):
//   BiasAddGrad  bias_op_gpu.cu.cc:93-242 (ThenMemZero + shared/global atomicAdd, order varies)
//                -> two-stage ordered column reduction, no atomics, bit-reproducible
//   Softmax      softmax_op_gpu.cu.cc:32-44 (SoftmaxEigenImpl = 4 Eigen kernels + 2 temporaries)
//                -> one kernel, one read + one write of the matrix
//   Xent         xent_op_gpu.cu.cc (XentEigenImpl, xent_op.h:47-113) -> one kernel
//   ArgMax       argmax_op_gpu.cu.cc (Eigen argmax reducer, argmax_op.h:29-42)
#include <atomic>
#include <cfloat>
#include <cuda_bf16.h>
#include <algorithm>

#include "b200_internal.h"
#include "ordered_reduce.cuh"

namespace b200 {

__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename T>
__device__ __forceinline__ float ldf(const T* p);
template <>
__device__ __forceinline__ float ldf<float>(const float* p) {
  return __ldg(p);
}
template <>
__device__ __forceinline__ float ldf<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <typename T>
__device__ __forceinline__ void stf(T* p, float v);
template <>
__device__ __forceinline__ void stf<float>(float* p, float v) {
  *p = v;
}
template <>
__device__ __forceinline__ void stf<__nv_bfloat16>(__nv_bfloat16* p, float v) {
  *p = __float2bfloat16_rn(v);
}

// Load batching.  ptxas schedules for register pressure and interleaves the adds with a batch of
// independent 16-byte loads so that only ~3 stay in flight per thread (checked in SASS; neither
// unrolling nor volatile asm changes it).  cp.async has no destination registers: a thread issues
// its whole batch into a private shared-memory slot per load and waits once, i.e. one memory
// latency per batch.  src_bytes = 0 zero-fills the slot (rows past the end contribute +0).
__device__ __forceinline__ void cp_async16_zfill(void* smem_dst, const void* gsrc, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(
                   static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))),
               "l"(gsrc), "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
}

// ================================================================== BiasAddGrad
// Stage 1: block (32, 8).  Columns are processed in vectors of VEC elements (16 bytes when the
// channel count allows).  W = channels / VEC vector-columns.  If W >= 32 a CTA owns 32
// vector-columns; if W < 32 the spare lanes fold extra rows (fold = 32 / W) so small channel
// counts (LeNet: 32, 64, 10) still use every lane.  Each CTA reduces a contiguous chunk of rows
// and writes one partial row; stage 2 adds the partial rows in chunk order.
// Single-launch form: the CTA that finishes a column tile LAST (ticket from a self-resetting
// counter) adds that tile's partial rows in the same fixed order as bias_grad_stage2, so the result
// is bit-identical to the two-kernel form and independent of which CTA happens to be last.
constexpr int kBiasGradSlots = 32, kBiasGradMaxTiles = 1024;
__device__ unsigned int g_bias_grad_tickets[kBiasGradSlots][kBiasGradMaxTiles];

template <typename T, int VEC, typename TOut = T>
__global__ void __launch_bounds__(256)
bias_grad_stage1(const T* __restrict__ g, float* __restrict__ partial, long long rows,
                 int channels, int rows_per_chunk, TOut* __restrict__ fused_out = nullptr,
                 unsigned int* __restrict__ tickets = nullptr) {
  pdl_prologue();
  const int W = channels / VEC;
  const int wt = W < 32 ? W : 32;        // vector-columns handled per CTA
  const int fold = W < 32 ? 32 / W : 1;  // rows covered by one warp-row
  const int x = threadIdx.x, y = threadIdx.y;
  const int cv = blockIdx.x * 32 + (x % wt);
  const int sub = x / wt;
  const bool active = sub < fold && cv < W;
  const long long r0 = (long long)blockIdx.y * rows_per_chunk;
  long long r1 = r0 + rows_per_chunk;
  if (r1 > rows) r1 = rows;
  float acc[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
  __shared__ uint4 stage[VEC > 1 ? 8 : 1][256];
  const int tid = y * 32 + x;
  if (active) {
    // Up to eight independent row loads in flight per thread (rows r, r + step, ...): with the
    // plan's 8 rows per thread the whole chunk is ONE batch, i.e. one HBM latency.  Rows past the
    // chunk contribute +0; the adds run in ascending row order whatever the batch size.
    constexpr int U = 8;
    const long long step = 8 * fold;
    for (long long r = r0 + y * fold + sub; r < r1; r += U * step) {
      if (VEC == 1) {
        float v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long rr = r + u * step;
          v[u] = rr < r1 ? ldf<T>(g + rr * channels + cv) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) acc[0] += v[u];
      } else {
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const long long rr = r + u * step;
          cp_async16_zfill(&stage[u][tid],
                           g + (rr < r1 ? rr : r1 - 1) * channels + (long long)cv * VEC,
                           rr < r1 ? 16 : 0);
        }
        cp_async_wait_all();
        uint4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = stage[u][tid];  // own slots only: no CTA barrier
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
          if (sizeof(T) == 4) {
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i % VEC] += __uint_as_float(w[i]);
          } else {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              acc[(2 * i) % VEC] += __uint_as_float(w[i] << 16);
              acc[(2 * i + 1) % VEC] += __uint_as_float(w[i] & 0xFFFF0000u);
            }
          }
        }
      }
    }
  }
  __shared__ float sm[8][32][VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) sm[y][x][j] = active ? acc[j] : 0.f;
  __syncthreads();
  if (y == 0 && sub == 0 && cv < W) {
    float tot[VEC];
#pragma unroll
    for (int j = 0; j < VEC; ++j) tot[j] = 0.f;
    for (int yy = 0; yy < 8; ++yy)
      for (int s = 0; s < fold; ++s)
#pragma unroll
        for (int j = 0; j < VEC; ++j) tot[j] += sm[yy][x + s * wt][j];
    float* dst = partial + (long long)blockIdx.y * channels + (long long)cv * VEC;
#pragma unroll
    for (int j = 0; j < VEC; ++j) dst[j] = tot[j];
    __threadfence();  // publish this CTA's partial row before taking a ticket
  }
  if (fused_out == nullptr) return;
  __shared__ bool is_last;
  __syncthreads();
  if (x == 0 && y == 0) is_last = atomicAdd(&tickets[blockIdx.x], 1u) == gridDim.y - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  const int nchunks = gridDim.y;
  float tot[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) tot[j] = 0.f;
  if (sub == 0 && cv < W) {
    // eight partial rows in flight per thread (independent loads, ordered adds), 16-byte loads
    // when the row is vectorised
    constexpr int U2 = 8;
    for (int k0 = y; k0 < nchunks; k0 += 8 * (VEC % 4 == 0 ? U2 / (VEC / 4 > 0 ? VEC / 4 : 1) : U2)) {
      if (VEC % 4 == 0) {
        constexpr int Q = VEC % 4 == 0 ? VEC / 4 : 1;  // 16-byte loads per partial row
        constexpr int RB = U2 / Q;                       // partial rows per batch (8 slots)
#pragma unroll
        for (int u = 0; u < RB; ++u) {
          const int k = k0 + 8 * u;
          const float* src =
              partial + (long long)(k < nchunks ? k : nchunks - 1) * channels + (long long)cv * VEC;
#pragma unroll
          for (int q = 0; q < Q; ++q)
            cp_async16_zfill(&stage[u * Q + q][tid], src + 4 * q, k < nchunks ? 16 : 0);
        }
        cp_async_wait_all();
#pragma unroll
        for (int u = 0; u < RB; ++u)
#pragma unroll
          for (int q = 0; q < Q; ++q) {
            const uint4 t = stage[u * Q + q][tid];
            tot[(4 * q) % VEC] += __uint_as_float(t.x);
            tot[(4 * q + 1) % VEC] += __uint_as_float(t.y);
            tot[(4 * q + 2) % VEC] += __uint_as_float(t.z);
            tot[(4 * q + 3) % VEC] += __uint_as_float(t.w);
          }
      } else {
#pragma unroll
        for (int u = 0; u < U2; ++u) {
          const int k = k0 + 8 * u;
          if (k < nchunks) {
            const float* src = partial + (long long)k * channels + (long long)cv * VEC;
#pragma unroll
            for (int j = 0; j < VEC; ++j) tot[j] += __ldcg(src + j);
          }
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < VEC; ++j) sm[y][x][j] = tot[j];
  __syncthreads();
  if (y == 0 && sub == 0 && cv < W) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) {
      float t = 0.f;
      for (int yy = 0; yy < 8; ++yy) t += sm[yy][x][j];
      stf<TOut>(fused_out + (long long)cv * VEC + j, t);
    }
  }
  if (x == 0 && y == 0) tickets[blockIdx.x] = 0;  // ready for the next launch that uses this slot
}
// Stage 2: out[c] = sum over chunks (ascending); block (32, 8), 8-way strided then ordered merge.
template <typename T>
__global__ void __launch_bounds__(256)
bias_grad_stage2(const float* __restrict__ partial, T* __restrict__ out, int nchunks,
                 int channels) {
  pdl_prologue();
  const int c = blockIdx.x * 32 + threadIdx.x;
  float acc = 0.f;
  if (c < channels)
    for (int k = threadIdx.y; k < nchunks; k += 8) acc += partial[(long long)k * channels + c];
  __shared__ float sm[8][33];
  sm[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c < channels) {
    float t = 0.f;
    for (int yy = 0; yy < 8; ++yy) t += sm[yy][threadIdx.x];
    stf<T>(out + c, t);
  }
}

struct BiasGradPlan {
  int vec, col_tiles, nchunks, rows_per_chunk;
};
static BiasGradPlan plan_bias_grad(int dtype, long long rows, long long channels, bool aligned) {
  BiasGradPlan p;
  const int v16 = dtype == B200_DT_FLOAT ? 4 : 8;
  p.vec = (aligned && channels % v16 == 0) ? v16 : 1;
  const long long W = channels / p.vec;
  p.col_tiles = (int)((W + 31) / 32);
  const int fold = W < 32 ? (int)(32 / W) : 1;
  // Eight rows per thread = one batch of independent 16-byte loads (one HBM latency) per chunk,
  // and a second stage of nchunks / 8 partial rows per thread, again one batch for <= 64 chunks.
  // More rows than 256 such chunks: the chunks grow instead (the ordered second stage stays short).
  // B200TF_BIAS_GRAD_ROWS_PER_THREAD is a tuning knob for tools/op_bench.py.
  static const int rows_per_thread = [] {
    const char* v = getenv("B200TF_BIAS_GRAD_ROWS_PER_THREAD");
    const int n = v ? atoi(v) : 0;
    return n > 0 ? n : 8;
  }();
  const long long chunk_rows = 8LL * fold * rows_per_thread;
  long long want = (rows + chunk_rows - 1) / chunk_rows;
  if (want > 256) want = 256;
  if (want < 1) want = 1;
  p.rows_per_chunk = (int)((rows + want - 1) / want);
  p.nchunks = (int)((rows + p.rows_per_chunk - 1) / p.rows_per_chunk);
  return p;
}

// ================================================================== BiasAddGrad, NCHW
// The tensor is [batch][channels][image]; out[c] = sum over batch and image (BiasGradNCHW_SharedAtomics,
// bias_op_gpu.cu.cc:140-188, which accumulates with atomics).  Here: one warp per (plane, chunk of
// <= kNchwChunk contiguous elements) -- 16-byte loads when the image allows, lane-strided so a warp
// reads 512 contiguous bytes per step -- folds with shuffles and writes one fp32 partial at
// [c][n * chunks + k]; one CTA per channel then adds that channel's partials in index order.
// Fixed association everywhere: bit-reproducible.
constexpr int kNchwChunk = 4096;

template <typename T, bool kVec>
__global__ void __launch_bounds__(256)
bias_grad_nchw_stage1(const T* __restrict__ g, float* __restrict__ partial, long long items,
                      int channels, long long image, int chunks, long long per_channel) {
  pdl_prologue();
  constexpr int VEC = 16 / (int)sizeof(T);
  const int lane = threadIdx.x & 31;
  const long long item = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (item >= items) return;
  const long long plane = item / chunks;
  const int k = (int)(item - plane * chunks);
  const long long n = plane / channels;
  const int c = (int)(plane - n * channels);
  const long long e0 = (long long)k * kNchwChunk;
  long long e1 = e0 + kNchwChunk;
  if (e1 > image) e1 = image;
  const T* src = g + plane * image;
  float acc = 0.f;
  if (kVec) {
    for (long long e = e0 + (long long)lane * VEC; e < e1; e += 32 * VEC) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(src + e));
      const uint32_t w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (sizeof(T) == 4) {
          acc += __uint_as_float(w[i]);
        } else {
          acc += __uint_as_float(w[i] << 16);
          acc += __uint_as_float(w[i] & 0xFFFF0000u);
        }
      }
    }
  } else {
    for (long long e = e0 + lane; e < e1; e += 32) acc += ldf<T>(src + e);
  }
  acc = warp_sum(acc);
  if (lane == 0) partial[(long long)c * per_channel + n * chunks + k] = acc;
}

template <typename T>
__global__ void __launch_bounds__(256)
bias_grad_nchw_stage2(const float* __restrict__ partial, T* __restrict__ out, long long per_channel) {
  pdl_prologue();
  const float* src = partial + (long long)blockIdx.x * per_channel;
  float acc = 0.f;
  for (long long i = threadIdx.x; i < per_channel; i += 256) acc += src[i];
  __shared__ float sm[256];
  sm[threadIdx.x] = acc;
  __syncthreads();
  for (int off = 128; off > 0; off >>= 1) {
    if ((int)threadIdx.x < off) sm[threadIdx.x] += sm[threadIdx.x + off];
    __syncthreads();
  }
  if (threadIdx.x == 0) stf<T>(out + blockIdx.x, sm[0]);
}

// ================================================================== flat BiasAddGrad (+ ReluGrad)
// For channel counts whose 16-byte vector columns divide a warp (G = C / VEC in {1, 2, .., 32}:
// the conv layers' 32 / 64 channels): the [rows, C] matrix is streamed as ONE flat array of
// 16-byte vectors.  The grid stride is a multiple of G, so a thread always meets the same column
// group (lane % G) and simply accumulates -- fully coalesced loads, several in flight, no index
// arithmetic.  Lanes of a column group are folded with shuffles, warps through shared memory, CTAs
// through an ordered last-ticket pass (fixed order: deterministic, no atomics on the data).
// kFused: the matrix is produced on the fly as ReluGrad(g, features) = g * (features > 0)
// (relu_op_functor.h:44-60) and written to `dy`: the ReluGrad -> BiasAddGrad pair of a conv layer's
// backward pass reads g and features once and writes dy once instead of re-reading dy.
__device__ unsigned int g_flat_bias_grad_tickets[kBiasGradSlots];

template <typename T, bool kFused>
__global__ void __launch_bounds__(256)
flat_bias_grad_kernel(const T* __restrict__ g, const T* __restrict__ features, T* __restrict__ dy,
                      float* __restrict__ partial, T* __restrict__ out, long long nvec, int G,
                      unsigned int* __restrict__ ticket) {
  pdl_prologue();
  constexpr int VEC = 16 / (int)sizeof(T);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long stride = (long long)gridDim.x * 256;
  float acc[VEC];
#pragma unroll
  for (int j = 0; j < VEC; ++j) acc[j] = 0.f;
  const uint4* gv = reinterpret_cast<const uint4*>(g);
  const uint4* fv = reinterpret_cast<const uint4*>(features);
  uint4* dv = reinterpret_cast<uint4*>(dy);
  auto consume = [&](uint4 x, uint4 f, long long v) {
    uint32_t xs[4] = {x.x, x.y, x.z, x.w};
    if (kFused) {
      const uint32_t fs[4] = {f.x, f.y, f.z, f.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (sizeof(T) == 4) {
          xs[i] = __uint_as_float(fs[i]) > 0.f ? xs[i] : __float_as_uint(__uint_as_float(xs[i]) * 0.f);
        } else {  // two bf16 per word: the mask is taken per element
          const float lo = __uint_as_float(xs[i] << 16), hi = __uint_as_float(xs[i] & 0xFFFF0000u);
          const bool klo = __uint_as_float(fs[i] << 16) > 0.f;
          const bool khi = __uint_as_float(fs[i] & 0xFFFF0000u) > 0.f;
          const uint32_t wlo = klo ? (xs[i] & 0xFFFFu) : (__float_as_uint(lo * 0.f) >> 16);
          const uint32_t whi = khi ? (xs[i] & 0xFFFF0000u) : (__float_as_uint(hi * 0.f) & 0xFFFF0000u);
          xs[i] = wlo | whi;
        }
      }
      dv[v] = make_uint4(xs[0], xs[1], xs[2], xs[3]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (sizeof(T) == 4) {
        acc[i % VEC] += __uint_as_float(xs[i]);
      } else {
        acc[(2 * i) % VEC] += __uint_as_float(xs[i] << 16);
        acc[(2 * i + 1) % VEC] += __uint_as_float(xs[i] & 0xFFFF0000u);
      }
    }
  };
  long long v = (long long)blockIdx.x * 256 + threadIdx.x;
  for (; v + 3 * stride < nvec; v += 4 * stride) {  // four independent 16-byte loads in flight
    uint4 x[4], f[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      x[u] = __ldg(gv + v + u * stride);
      if (kFused) f[u] = __ldg(fv + v + u * stride);
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) consume(x[u], kFused ? f[u] : x[u], v + u * stride);
  }
  for (; v < nvec; v += stride) {
    const uint4 x = __ldg(gv + v);
    consume(x, kFused ? __ldg(fv + v) : x, v);
  }
  // lanes with the same lane % G hold the same column group
  for (int off = G; off < 32; off <<= 1) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) acc[j] += __shfl_xor_sync(0xffffffffu, acc[j], off);
  }
  __shared__ float sm[8][32][VEC];
  if (lane < G) {
#pragma unroll
    for (int j = 0; j < VEC; ++j) sm[warp][lane][j] = acc[j];
  }
  __syncthreads();
  const int C = G * VEC;
  if ((int)threadIdx.x < C) {
    const int cg = threadIdx.x / VEC, j = threadIdx.x % VEC;
    float t = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += sm[w][cg][j];
    partial[(long long)blockIdx.x * C + threadIdx.x] = t;
    __threadfence();
  }
  __shared__ bool is_last;
  __syncthreads();
  if (threadIdx.x == 0) is_last = atomicAdd(ticket, 1u) == gridDim.x - 1;
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  // ordered final pass over the per-CTA partial rows (ordered_reduce.cuh)
  __shared__ uint4 slots[8 * 256];
  __shared__ float flat[256 * 4];
  const float tot = ordered_partial_sum(partial, (int)gridDim.x, C, slots, flat);
  if ((int)threadIdx.x < C) stf<T>(out + threadIdx.x, tot);
  if (threadIdx.x == 0) *ticket = 0;  // ready for the next launch that uses this slot
}

struct FlatBiasGradPlan {
  bool ok;
  int G, blocks;
  long long nvec;
};
static FlatBiasGradPlan plan_flat_bias_grad(int dtype, long long rows, long long channels) {
  FlatBiasGradPlan p{false, 0, 0, 0};
  const int vec = dtype == B200_DT_FLOAT ? 4 : 8;
  if (channels % vec != 0) return p;
  const long long G = channels / vec;
  if (G < 1 || G > 32 || (G & (G - 1)) != 0) return p;
  p.G = (int)G;
  p.nvec = rows * G;
  long long blocks = (p.nvec + 256 * 8 - 1) / (256 * 8);  // >= 8 vectors per thread
  const long long cap = 4LL * sm_count();
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  p.blocks = (int)blocks;
  p.ok = true;
  return p;
}
template <typename T>
static int launch_flat_bias_grad(const FlatBiasGradPlan& p, const void* g, const void* features,
                                 void* dy, void* out, void* workspace, cudaStream_t s) {
  static std::atomic<unsigned> next_slot{0};
  unsigned int* base = nullptr;
  if (cudaGetSymbolAddress(reinterpret_cast<void**>(&base), g_flat_bias_grad_tickets) != cudaSuccess)
    return check_launch("flat_bias_grad");
  unsigned int* ticket = base + next_slot.fetch_add(1) % kBiasGradSlots;
  float* partial = static_cast<float*>(workspace);
  if (features != nullptr)
    launch_pdl(flat_bias_grad_kernel<T, true>, dim3(p.blocks), dim3(256), 0, s,
               static_cast<const T*>(g), static_cast<const T*>(features), static_cast<T*>(dy), partial,
               static_cast<T*>(out), p.nvec, p.G, ticket);
  else
    launch_pdl(flat_bias_grad_kernel<T, false>, dim3(p.blocks), dim3(256), 0, s,
               static_cast<const T*>(g), static_cast<const T*>(nullptr), static_cast<T*>(nullptr),
               partial, static_cast<T*>(out), p.nvec, p.G, ticket);
  note_launch();
  return check_launch("flat_bias_grad");
}

// ================================================================== Softmax family
// Row-per-warp, whole row held in registers: NV float4 (or 8 x bf16) per lane => cols <= 128*NV
// (or 256*NV).  One HBM read and one write of the matrix.
template <typename T, int NV, bool kLog>
__global__ void __launch_bounds__(256)
softmax_warp_kernel(const T* __restrict__ logits, T* __restrict__ out, long long rows, int cols) {
  pdl_prologue();
  constexpr int E = 16 / sizeof(T);  // elements per 16-byte vector
  const int lane = threadIdx.x & 31;
  // persistent: warps stride over rows (grid capped at ~8 CTAs/SM, no CTA wave transitions)
  for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows;
       row += (long long)gridDim.x * 8) {
  const T* x = logits + row * cols;
  float v[NV][E];
  float mx = -FLT_MAX;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c0 = (lane + 32 * j) * E;
    if (c0 < cols) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(x + c0));
      if (sizeof(T) == 4) {
        v[j][0] = __uint_as_float(q.x);
        v[j][1] = __uint_as_float(q.y);
        v[j][2 % E] = __uint_as_float(q.z);
        v[j][3 % E] = __uint_as_float(q.w);
      } else {
        const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          v[j][(2 * i) % E] = __uint_as_float(w[i] << 16);
          v[j][(2 * i + 1) % E] = __uint_as_float(w[i] & 0xFFFF0000u);
        }
      }
#pragma unroll
      for (int e = 0; e < E; ++e) mx = fmaxf(mx, v[j][e]);
    }
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c0 = (lane + 32 * j) * E;
    if (c0 < cols) {
#pragma unroll
      for (int e = 0; e < E; ++e) {
        v[j][e] -= mx;  // shifted logits
        const float ex = expf(v[j][e]);
        sum += ex;
        if (!kLog) v[j][e] = ex;
      }
    }
  }
  sum = warp_sum(sum);
  const float k = kLog ? logf(sum) : 1.f / sum;
  T* y = out + row * cols;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int c0 = (lane + 32 * j) * E;
    if (c0 < cols) {
      float r[E];
#pragma unroll
      for (int e = 0; e < E; ++e) r[e] = kLog ? v[j][e] - k : v[j][e] * k;
      uint4 q;
      if (sizeof(T) == 4) {
        q = make_uint4(__float_as_uint(r[0]), __float_as_uint(r[1]), __float_as_uint(r[2 % E]),
                       __float_as_uint(r[3 % E]));
      } else {
        uint32_t w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          __nv_bfloat162 h = __floats2bfloat162_rn(r[(2 * i) % E], r[(2 * i + 1) % E]);
          w[i] = *reinterpret_cast<uint32_t*>(&h);
        }
        q = make_uint4(w[0], w[1], w[2], w[3]);
      }
      *reinterpret_cast<uint4*>(y + c0) = q;
    }
  }
  }  // row loop
}

// Generic fallback: one CTA (256 threads) per row, three passes over the row (L1/L2 resident),
// any column count / alignment.  Also carries the xent variant.
__device__ __forceinline__ float block_reduce(float v, bool is_max, float* sm) {
  v = is_max ? warp_max(v) : warp_sum(v);
  const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
  __syncthreads();
  if (l == 0) sm[w] = v;
  __syncthreads();
  float r = is_max ? -FLT_MAX : 0.f;
  for (int i = 0; i < 8; ++i) r = is_max ? fmaxf(r, sm[i]) : r + sm[i];
  return r;
}
template <typename T, bool kLog>
__global__ void __launch_bounds__(256)
softmax_block_kernel(const T* __restrict__ logits, T* __restrict__ out, int cols) {
  pdl_prologue();
  __shared__ float sm[8];
  const T* x = logits + (long long)blockIdx.x * cols;
  T* y = out + (long long)blockIdx.x * cols;
  float mx = -FLT_MAX;
  for (int c = threadIdx.x; c < cols; c += 256) mx = fmaxf(mx, ldf<T>(x + c));
  mx = block_reduce(mx, true, sm);
  float sum = 0.f;
  for (int c = threadIdx.x; c < cols; c += 256) sum += expf(ldf<T>(x + c) - mx);
  sum = block_reduce(sum, false, sm);
  const float k = kLog ? logf(sum) : 1.f / sum;
  for (int c = threadIdx.x; c < cols; c += 256) {
    const float s = ldf<T>(x + c) - mx;
    stf<T>(y + c, kLog ? s - k : expf(s) * k);
  }
}
// loss[r] = sum_c labels * (log(sum) - shifted); backprop = exp(shifted) / sum - labels
template <typename T>
__global__ void __launch_bounds__(256)
xent_block_kernel(const T* __restrict__ logits, const T* __restrict__ labels, T* __restrict__ loss,
                  T* __restrict__ backprop, int cols, const float* __restrict__ bp_scale) {
  pdl_prologue();
  __shared__ float sm[8];
  const float sc = bp_scale ? __ldg(bp_scale) : 1.0f;  // x * 1.0f is exact: unscaled unchanged
  const T* x = logits + (long long)blockIdx.x * cols;
  const T* l = labels + (long long)blockIdx.x * cols;
  T* bp = backprop + (long long)blockIdx.x * cols;
  float mx = -FLT_MAX;
  for (int c = threadIdx.x; c < cols; c += 256) mx = fmaxf(mx, ldf<T>(x + c));
  mx = block_reduce(mx, true, sm);
  float sum = 0.f;
  for (int c = threadIdx.x; c < cols; c += 256) sum += expf(ldf<T>(x + c) - mx);
  sum = block_reduce(sum, false, sm);
  const float ls = logf(sum);
  float acc = 0.f;
  for (int c = threadIdx.x; c < cols; c += 256) {
    const float s = ldf<T>(x + c) - mx;
    const float lab = ldf<T>(l + c);
    acc += lab * (ls - s);
    stf<T>(bp + c, (expf(s) / sum - lab) * sc);
  }
  acc = block_reduce(acc, false, sm);
  if (threadIdx.x == 0) stf<T>(loss + blockIdx.x, acc);
}
// Row-per-warp xent for cols <= 1024 (the MLP's 1024-class logits, LeNet's 10 classes).
template <typename T>
__global__ void __launch_bounds__(256)
xent_warp_kernel(const T* __restrict__ logits, const T* __restrict__ labels, T* __restrict__ loss,
                 T* __restrict__ backprop, long long rows, int cols,
                 const float* __restrict__ bp_scale) {
  pdl_prologue();
  const float sc = bp_scale ? __ldg(bp_scale) : 1.0f;
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const T* x = logits + row * cols;
  const T* l = labels + row * cols;
  T* bp = backprop + row * cols;
  float v[32], lab[32];
  float mx = -FLT_MAX;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const int c = lane + 32 * j;
    if (c < cols) {
      v[j] = ldf<T>(x + c);
      lab[j] = ldf<T>(l + c);
      mx = fmaxf(mx, v[j]);
    }
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (lane + 32 * j < cols) {
      v[j] -= mx;
      sum += expf(v[j]);
    }
  sum = warp_sum(sum);
  const float ls = logf(sum);
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) {
    const int c = lane + 32 * j;
    if (c < cols) {
      acc += lab[j] * (ls - v[j]);
      stf<T>(bp + c, (expf(v[j]) / sum - lab[j]) * sc);
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) stf<T>(loss + row, acc);
}

// fp32, cols % 4 == 0, cols <= 128 * NV: 16-byte loads, whole row of logits and labels in registers.
template <int NV>
__global__ void __launch_bounds__(256)
xent_warp_vec_kernel(const float* __restrict__ logits, const float* __restrict__ labels,
                     float* __restrict__ loss, float* __restrict__ backprop, long long rows,
                     int cols, const float* __restrict__ bp_scale) {
  pdl_prologue();
  const float sc = bp_scale ? __ldg(bp_scale) : 1.0f;
  const int lane = threadIdx.x & 31;
  for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows;
       row += (long long)gridDim.x * 8) {
  const float4* x = reinterpret_cast<const float4*>(logits + row * cols);
  const float4* l = reinterpret_cast<const float4*>(labels + row * cols);
  float4* bp = reinterpret_cast<float4*>(backprop + row * cols);
  const int nvec = cols >> 2;
  float4 v[NV], lab[NV], ex[NV];
  float mx = -FLT_MAX;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      v[j] = __ldg(x + i);
      lab[j] = __ldg(l + i);
      mx = fmaxf(mx, fmaxf(fmaxf(v[j].x, v[j].y), fmaxf(v[j].z, v[j].w)));
    }
  }
  mx = warp_max(mx);
  float sum = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j)
    if (lane + 32 * j < nvec) {
      v[j].x -= mx;
      v[j].y -= mx;
      v[j].z -= mx;
      v[j].w -= mx;
      // exp is evaluated once per element and kept for the backprop pass
      ex[j] = make_float4(expf(v[j].x), expf(v[j].y), expf(v[j].z), expf(v[j].w));
      sum += ex[j].x + ex[j].y + ex[j].z + ex[j].w;
    }
  sum = warp_sum(sum);
  const float ls = logf(sum);
  float acc = 0.f;
#pragma unroll
  for (int j = 0; j < NV; ++j) {
    const int i = lane + 32 * j;
    if (i < nvec) {
      acc += lab[j].x * (ls - v[j].x) + lab[j].y * (ls - v[j].y) + lab[j].z * (ls - v[j].z) +
             lab[j].w * (ls - v[j].w);
      float4 o;
      o.x = (ex[j].x / sum - lab[j].x) * sc;
      o.y = (ex[j].y / sum - lab[j].y) * sc;
      o.z = (ex[j].z / sum - lab[j].z) * sc;
      o.w = (ex[j].w / sum - lab[j].w) * sc;
      bp[i] = o;
    }
  }
  acc = warp_sum(acc);
  if (lane == 0) loss[row] = acc;
  }  // row loop
}

// bf16, cols % 8 == 0, cols <= 256 * NV: 16-byte loads (8 elements), the row of logits and labels in
// registers as fp32; same arithmetic as xent_warp_kernel<bf16> (fp32 math, one rounding per output).
template <int NV>
__global__ void __launch_bounds__(256)
xent_warp_vec_bf16_kernel(const __nv_bfloat16* __restrict__ logits,
                          const __nv_bfloat16* __restrict__ labels, __nv_bfloat16* __restrict__ loss,
                          __nv_bfloat16* __restrict__ backprop, long long rows, int cols) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const int nvec = cols >> 3;
  for (long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5); row < rows;
       row += (long long)gridDim.x * 8) {
    const uint4* x = reinterpret_cast<const uint4*>(logits + row * cols);
    const uint4* l = reinterpret_cast<const uint4*>(labels + row * cols);
    uint4* bp = reinterpret_cast<uint4*>(backprop + row * cols);
    float v[NV][8], lab[NV][8];
    float mx = -FLT_MAX;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec) {
        const uint4 a = __ldg(x + i), b = __ldg(l + i);
        const uint32_t aw[4] = {a.x, a.y, a.z, a.w}, bw[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          v[j][2 * q] = __uint_as_float(aw[q] << 16);
          v[j][2 * q + 1] = __uint_as_float(aw[q] & 0xFFFF0000u);
          lab[j][2 * q] = __uint_as_float(bw[q] << 16);
          lab[j][2 * q + 1] = __uint_as_float(bw[q] & 0xFFFF0000u);
          mx = fmaxf(mx, fmaxf(v[j][2 * q], v[j][2 * q + 1]));
        }
      }
    }
    mx = warp_max(mx);
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j)
      if (lane + 32 * j < nvec) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          v[j][q] -= mx;
          sum += expf(v[j][q]);
        }
      }
    sum = warp_sum(sum);
    const float ls = logf(sum);
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < NV; ++j) {
      const int i = lane + 32 * j;
      if (i < nvec) {
        uint32_t ow[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          acc += lab[j][2 * q] * (ls - v[j][2 * q]);
          acc += lab[j][2 * q + 1] * (ls - v[j][2 * q + 1]);
          const __nv_bfloat16 lo = __float2bfloat16_rn(expf(v[j][2 * q]) / sum - lab[j][2 * q]);
          const __nv_bfloat16 hi =
              __float2bfloat16_rn(expf(v[j][2 * q + 1]) / sum - lab[j][2 * q + 1]);
          ow[q] = (uint32_t)__bfloat16_as_ushort(lo) | ((uint32_t)__bfloat16_as_ushort(hi) << 16);
        }
        bp[i] = make_uint4(ow[0], ow[1], ow[2], ow[3]);
      }
    }
    acc = warp_sum(acc);
    if (lane == 0) loss[row] = __float2bfloat16_rn(acc);
  }
}

// ================================================================== ArgMax
template <typename T>
__device__ __forceinline__ T arg_lowest();
template <>
__device__ __forceinline__ float arg_lowest<float>() {
  return -FLT_MAX;
}
template <>
__device__ __forceinline__ int32_t arg_lowest<int32_t>() {
  return INT32_MIN;
}
template <>
__device__ __forceinline__ int64_t arg_lowest<int64_t>() {
  return INT64_MIN;
}
// inner == 1: one warp per row; (value, index) butterfly, lower index wins ties.
template <typename T>
__global__ void __launch_bounds__(256)
argmax_last_axis_kernel(const T* __restrict__ in, int64_t* __restrict__ out, long long outer,
                        long long axis) {
  pdl_prologue();
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= outer) return;
  const T* x = in + row * axis;
  T bv = arg_lowest<T>();
  long long bi = 0;  // Eigen's reducer starts at (index 0, lowest) and needs strict > to move
  for (long long a = lane; a < axis; a += 32) {
    const T v = x[a];
    if (v > bv) {
      bv = v;
      bi = a;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const T ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const long long oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (ov > bv || (ov == bv && oi < bi)) {
      bv = ov;
      bi = oi;
    }
  }
  // a lane that saw no element > lowest keeps index 0; with ties on lowest the smallest lane
  // index wins, and index 0 is the smallest possible
  if (lane == 0) out[row] = bi;
}
// general: one thread per (outer, inner) walks the axis; coalesced across inner.
template <typename T>
__global__ void __launch_bounds__(256)
argmax_strided_kernel(const T* __restrict__ in, int64_t* __restrict__ out, long long outer,
                      long long axis, long long inner) {
  pdl_prologue();
  const long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= outer * inner) return;
  const long long o = i / inner, k = i - o * inner;
  const T* x = in + o * axis * inner + k;
  T bv = arg_lowest<T>();
  long long bi = 0;
  for (long long a = 0; a < axis; ++a) {
    const T v = x[a * inner];
    if (v > bv) {
      bv = v;
      bi = a;
    }
  }
  out[i] = bi;
}

// ================================================================== deterministic sum
__global__ void __launch_bounds__(256)
sum_stage1(const float* __restrict__ in, float* __restrict__ partial, long long n) {
  pdl_prologue();
  __shared__ float sm[8];
  float acc = 0.f;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += 256LL * gridDim.x)
    acc += in[i];
  acc = block_reduce(acc, false, sm);
  if (threadIdx.x == 0) partial[blockIdx.x] = acc;
}
__global__ void __launch_bounds__(256)
sum_stage2(const float* __restrict__ partial, float* __restrict__ out, int n, float scale) {
  pdl_prologue();
  __shared__ float sm[8];
  float acc = 0.f;
  for (int i = threadIdx.x; i < n; i += 256) acc += partial[i];
  acc = block_reduce(acc, false, sm);
  if (threadIdx.x == 0) out[0] = acc * scale;
}
// single CTA variant when n is small: no scratch needed
__global__ void __launch_bounds__(256)
sum_single(const float* __restrict__ in, float* __restrict__ out, long long n, float scale) {
  pdl_prologue();
  __shared__ float sm[8];
  float acc = 0.f;
  for (long long i = threadIdx.x; i < n; i += 256) acc += in[i];
  acc = block_reduce(acc, false, sm);
  if (threadIdx.x == 0) out[0] = acc * scale;
}

// General Sum / Mean over one contiguous run of axes: in viewed as [outer, reduce, inner],
// out[o, i] = scale * sum_r in[o, r, i], fp32 accumulation in a fixed order (deterministic).
// (the reference: ReductionOp<Device, T, Reducer>, core/kernels/reduction_ops_common.h, which
// collapses adjacent reduced / kept axes the same way before handing Eigen a 2-D / 3-D reduce)
//   inner == 1: one CTA per outer row, 256 threads stride over `reduce`, tree in the block.
//   inner  > 1: a CTA owns 32 inner columns x 8 row groups; threads of a warp read consecutive
//               columns (coalesced), the 8 groups are combined through shared memory.
template <typename T>
__global__ void __launch_bounds__(256)
reduce_rows_kernel(const T* __restrict__ in, T* __restrict__ out, long long reduce, float scale) {
  pdl_prologue();
  __shared__ float sm[8];
  const T* x = in + (long long)blockIdx.x * reduce;
  float acc = 0.f;
  for (long long i = threadIdx.x; i < reduce; i += 256) acc += ldf<T>(x + i);
  acc = block_reduce(acc, false, sm);
  if (threadIdx.x == 0) stf<T>(out + blockIdx.x, acc * scale);
}
template <typename T>
__global__ void __launch_bounds__(256)
reduce_mid_kernel(const T* __restrict__ in, T* __restrict__ out, long long outer, long long reduce,
                  long long inner, float scale) {
  pdl_prologue();
  __shared__ float sm[8][32];
  const int x = threadIdx.x & 31, y = threadIdx.x >> 5;
  const long long col = (long long)blockIdx.x * 32 + x;
  // grid-stride over `outer` (gridDim.y is capped at 65535); each (outer, column) is summed in the
  // same order whatever the grid
  for (long long o = blockIdx.y; o < outer; o += gridDim.y) {
    const T* base = in + o * reduce * inner;
    float acc = 0.f;
    if (col < inner)
      for (long long r = y; r < reduce; r += 8) acc += ldf<T>(base + r * inner + col);
    __syncthreads();  // the previous row's merge has read sm
    sm[y][x] = acc;
    __syncthreads();
    if (y == 0 && col < inner) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) t += sm[i][x];
      stf<T>(out + o * inner + col, t * scale);
    }
  }
}
template <typename T>
static int launch_reduce(const void* in, void* out, long long outer, long long reduce,
                         long long inner, float scale, cudaStream_t s) {
  const T* x = static_cast<const T*>(in);
  T* y = static_cast<T*>(out);
  if (inner == 1) {
    launch_pdl(reduce_rows_kernel<T>, dim3((unsigned)outer), dim3(256), 0, s, x, y, reduce, scale);
  } else {
    const unsigned gy = (unsigned)std::min<long long>(outer, 65535);
    launch_pdl(reduce_mid_kernel<T>, dim3((unsigned)((inner + 31) / 32), gy), dim3(256), 0, s, x, y,
               outer, reduce, inner, scale);
  }
  return B200_OK;
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

template <typename T>
static int launch_softmax(const void* logits, void* out, long long rows, int cols, bool log_sm,
                          cudaStream_t s) {
  constexpr int E = 16 / sizeof(T);
  const T* x = static_cast<const T*>(logits);
  T* y = static_cast<T*>(out);
  const bool vec = cols % E == 0 && aligned16(logits) && aligned16(out);
  const int nv = (cols + 32 * E - 1) / (32 * E);  // 16-byte vectors per lane
  unsigned wgrid = (unsigned)((rows + 7) / 8);
  if (wgrid > 8u * (unsigned)sm_count()) wgrid = 8u * (unsigned)sm_count();
#define SM_LAUNCH(NV)                                                                   \
  do {                                                                                  \
    if (log_sm)                                                                         \
      launch_pdl(softmax_warp_kernel<T, NV, true>, dim3(wgrid), dim3(256), 0, s, x, y, rows, cols);         \
    else                                                                                \
      launch_pdl(softmax_warp_kernel<T, NV, false>, dim3(wgrid), dim3(256), 0, s, x, y, rows, cols);        \
  } while (0)
  if (vec && nv <= 8) {
    if (nv <= 1)
      SM_LAUNCH(1);
    else if (nv <= 2)
      SM_LAUNCH(2);
    else if (nv <= 4)
      SM_LAUNCH(4);
    else
      SM_LAUNCH(8);
  } else {
    if (log_sm)
      launch_pdl(softmax_block_kernel<T, true>, dim3((unsigned)rows), dim3(256), 0, s, x, y, cols);
    else
      launch_pdl(softmax_block_kernel<T, false>, dim3((unsigned)rows), dim3(256), 0, s, x, y, cols);
  }
#undef SM_LAUNCH
  note_launch();
  return check_launch("b200_softmax");
}

}  // namespace b200

using namespace b200;

extern "C" {

size_t b200_bias_add_grad_workspace_bytes(int dtype, int64_t rows, int64_t channels) {
  if (rows <= 0 || channels <= 0) return 0;
  // alignment-independent upper bound: the scalar plan never needs more chunks than the vector one
  BiasGradPlan a = plan_bias_grad(dtype, rows, channels, true);
  BiasGradPlan b = plan_bias_grad(dtype, rows, channels, false);
  const int n = a.nchunks > b.nchunks ? a.nchunks : b.nchunks;
  size_t need = (size_t)n * (size_t)channels * sizeof(float);
  const FlatBiasGradPlan f = plan_flat_bias_grad(dtype, rows, channels);
  if (f.ok) need = std::max(need, (size_t)f.blocks * (size_t)channels * sizeof(float));
  return need;
}

size_t b200_bias_add_grad_nchw_workspace_bytes(int dtype, int64_t batch, int64_t channels,
                                               int64_t image) {
  (void)dtype;
  if (batch <= 0 || channels <= 0 || image <= 0) return 0;
  const int64_t chunks = (image + kNchwChunk - 1) / kNchwChunk;
  return (size_t)batch * (size_t)channels * (size_t)chunks * sizeof(float);
}

int b200_bias_add_grad_nchw(int dtype, const void* out_backprop, void* out, int64_t batch,
                            int64_t channels, int64_t image, void* workspace,
                            size_t workspace_bytes, void* stream) {
  if (batch < 0 || channels < 0 || image < 0 || channels > INT32_MAX) {
    set_last_error("b200_bias_add_grad_nchw: bad shape [%lld, %lld, %lld]", (long long)batch,
                   (long long)channels, (long long)image);
    return B200_INVALID_ARGUMENT;
  }
  if (dtype != B200_DT_FLOAT && dtype != B200_DT_BFLOAT16) {
    set_last_error("b200_bias_add_grad_nchw: unsupported dtype %d", dtype);
    return B200_UNIMPLEMENTED;
  }
  if (channels == 0) return B200_OK;
  const size_t esize = dtype == B200_DT_FLOAT ? 4 : 2;
  if (batch == 0 || image == 0)  // sum over nothing = 0 (bias_op.cc:206-209 zero-fills)
    return b200_memset_async(out, 0, (size_t)channels * esize, stream);
  int rc = require_device("b200_bias_add_grad_nchw");
  if (rc) return rc;
  const size_t need = b200_bias_add_grad_nchw_workspace_bytes(dtype, batch, channels, image);
  if (!workspace || workspace_bytes < need) {
    set_last_error("b200_bias_add_grad_nchw: workspace too small (%zu < %zu bytes)",
                   workspace_bytes, need);
    return B200_INVALID_ARGUMENT;
  }
  cudaStream_t s = as_stream(stream);
  const int chunks = (int)((image + kNchwChunk - 1) / kNchwChunk);
  const long long items = (long long)batch * channels * chunks;
  const long long blocks = (items + 7) / 8;
  if (blocks > INT32_MAX) {
    set_last_error("b200_bias_add_grad_nchw: too many planes");
    return B200_INVALID_ARGUMENT;
  }
  float* partial = static_cast<float*>(workspace);
  const int vec_elems = 16 / (int)esize;
  // kNchwChunk is a multiple of the vector width, so chunk starts stay 16-byte aligned
  const bool vec = image % vec_elems == 0 && aligned16(out_backprop);
  const long long per_channel = (long long)batch * chunks;
  if (dtype == B200_DT_FLOAT) {
    const float* gp = static_cast<const float*>(out_backprop);
    if (vec)
      launch_pdl(bias_grad_nchw_stage1<float, true>, dim3((unsigned)blocks), dim3(256), 0, s, gp,
                 partial, items, (int)channels, (long long)image, chunks, per_channel);
    else
      launch_pdl(bias_grad_nchw_stage1<float, false>, dim3((unsigned)blocks), dim3(256), 0, s, gp,
                 partial, items, (int)channels, (long long)image, chunks, per_channel);
    launch_pdl(bias_grad_nchw_stage2<float>, dim3((unsigned)channels), dim3(256), 0, s,
               (const float*)partial, static_cast<float*>(out), per_channel);
  } else {
    const __nv_bfloat16* gp = static_cast<const __nv_bfloat16*>(out_backprop);
    if (vec)
      launch_pdl(bias_grad_nchw_stage1<__nv_bfloat16, true>, dim3((unsigned)blocks), dim3(256), 0,
                 s, gp, partial, items, (int)channels, (long long)image, chunks, per_channel);
    else
      launch_pdl(bias_grad_nchw_stage1<__nv_bfloat16, false>, dim3((unsigned)blocks), dim3(256), 0,
                 s, gp, partial, items, (int)channels, (long long)image, chunks, per_channel);
    launch_pdl(bias_grad_nchw_stage2<__nv_bfloat16>, dim3((unsigned)channels), dim3(256), 0, s,
               (const float*)partial, static_cast<__nv_bfloat16*>(out), per_channel);
  }
  note_launch(2);
  return check_launch("b200_bias_add_grad_nchw");
}

size_t b200_relu_grad_bias_grad_workspace_bytes(int dtype, int64_t rows, int64_t channels) {
  return b200_bias_add_grad_workspace_bytes(dtype, rows, channels);
}

int b200_relu_grad_bias_grad(int dtype, const void* gradients, const void* features,
                             void* backprops, void* bias_grad, int64_t rows, int64_t channels,
                             void* workspace, size_t workspace_bytes, void* stream) {
  if (rows < 0 || channels < 0) {
    set_last_error("b200_relu_grad_bias_grad: negative size");
    return B200_INVALID_ARGUMENT;
  }
  if (dtype != B200_DT_FLOAT && dtype != B200_DT_BFLOAT16) {
    set_last_error("b200_relu_grad_bias_grad: unsupported dtype %d", dtype);
    return B200_UNIMPLEMENTED;
  }
  if (channels == 0) return B200_OK;
  const FlatBiasGradPlan f = plan_flat_bias_grad(dtype, rows, channels);
  const size_t need = f.ok ? (size_t)f.blocks * (size_t)channels * sizeof(float) : 0;
  static const bool off = getenv("B200TF_NO_FLAT_BIAS_GRAD") != nullptr;
  if (rows > 0 && f.ok && !off && workspace && workspace_bytes >= need && aligned16(gradients) &&
      aligned16(features) && aligned16(backprops)) {
    int rc = require_device("b200_relu_grad_bias_grad");
    if (rc) return rc;
    return dtype == B200_DT_FLOAT
               ? launch_flat_bias_grad<float>(f, gradients, features, backprops, bias_grad, workspace,
                                              as_stream(stream))
               : launch_flat_bias_grad<__nv_bfloat16>(f, gradients, features, backprops, bias_grad,
                                                      workspace, as_stream(stream));
  }
  // any other shape: the two library kernels back to back (same arithmetic)
  int rc = b200_relu_grad(dtype, gradients, features, backprops, rows * channels, stream);
  if (rc) return rc;
  return b200_bias_add_grad(dtype, backprops, bias_grad, rows, channels, workspace, workspace_bytes,
                            stream);
}

int b200_bias_add_grad(int dtype, const void* out_backprop, void* out, int64_t rows,
                       int64_t channels, void* workspace, size_t workspace_bytes, void* stream) {
  if (rows < 0 || channels < 0) {
    set_last_error("b200_bias_add_grad: negative size");
    return B200_INVALID_ARGUMENT;
  }
  if (dtype != B200_DT_FLOAT && dtype != B200_DT_BFLOAT16) {
    set_last_error("b200_bias_add_grad: unsupported dtype %d", dtype);
    return B200_UNIMPLEMENTED;
  }
  if (channels == 0) return B200_OK;
  int rc = require_device("b200_bias_add_grad");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  if (rows == 0)  // sum over nothing = 0 (bias_op.cc:206-209 zero-fills)
    return b200_memset_async(out, 0, (size_t)channels * (dtype == B200_DT_FLOAT ? 4 : 2), stream);
  if (channels > INT32_MAX) {
    set_last_error("b200_bias_add_grad: channels exceeds int32");
    return B200_INVALID_ARGUMENT;
  }
  {
    const FlatBiasGradPlan f = plan_flat_bias_grad(dtype, rows, channels);
    static const bool flat_off = getenv("B200TF_NO_FLAT_BIAS_GRAD") != nullptr;
    if (f.ok && !flat_off && aligned16(out_backprop) && workspace &&
        workspace_bytes >= (size_t)f.blocks * (size_t)channels * sizeof(float))
      return dtype == B200_DT_FLOAT
                 ? launch_flat_bias_grad<float>(f, out_backprop, nullptr, nullptr, out, workspace, s)
                 : launch_flat_bias_grad<__nv_bfloat16>(f, out_backprop, nullptr, nullptr, out,
                                                        workspace, s);
  }
  const BiasGradPlan p = plan_bias_grad(dtype, rows, channels, aligned16(out_backprop));
  const size_t need = (size_t)p.nchunks * (size_t)channels * sizeof(float);
  if (!workspace || workspace_bytes < need) {
    set_last_error("b200_bias_add_grad: workspace too small (%zu < %zu bytes)", workspace_bytes,
                   need);
    return B200_INVALID_ARGUMENT;
  }
  float* partial = static_cast<float*>(workspace);
  dim3 grid(p.col_tiles, p.nchunks), block(32, 8);
  static const bool two_kernels = getenv("B200TF_BIAS_GRAD_TWO_KERNELS") != nullptr;
  if (!two_kernels && p.col_tiles <= kBiasGradMaxTiles) {
    // Ticket counters: one row of a small ring per launch, so launches in flight on different
    // streams never share counters unless more than kBiasGradSlots of them overlap.
    static std::atomic<unsigned> next_slot{0};
    unsigned int* base = nullptr;
    if (cudaGetSymbolAddress(reinterpret_cast<void**>(&base), g_bias_grad_tickets) != cudaSuccess)
      return check_launch("b200_bias_add_grad");
    unsigned int* tickets =
        base + (size_t)(next_slot.fetch_add(1) % kBiasGradSlots) * kBiasGradMaxTiles;
    if (dtype == B200_DT_FLOAT) {
      const float* gp = static_cast<const float*>(out_backprop);
      float* op = static_cast<float*>(out);
      if (p.vec == 4)
        launch_pdl(bias_grad_stage1<float, 4>, dim3(grid), dim3(block), 0, s, gp, partial, rows, (int)channels,
                                                          p.rows_per_chunk, op, tickets);
      else
        launch_pdl(bias_grad_stage1<float, 1>, dim3(grid), dim3(block), 0, s, gp, partial, rows, (int)channels,
                                                          p.rows_per_chunk, op, tickets);
    } else {
      const __nv_bfloat16* gp = static_cast<const __nv_bfloat16*>(out_backprop);
      __nv_bfloat16* op = static_cast<__nv_bfloat16*>(out);
      if (p.vec == 8)
        launch_pdl(bias_grad_stage1<__nv_bfloat16, 8>, dim3(grid), dim3(block), 0, s, gp, partial, rows, (int)channels,
                                                                  p.rows_per_chunk, op, tickets);
      else
        launch_pdl(bias_grad_stage1<__nv_bfloat16, 1>, dim3(grid), dim3(block), 0, s, gp, partial, rows, (int)channels,
                                                                  p.rows_per_chunk, op, tickets);
    }
    note_launch(1);
    return check_launch("b200_bias_add_grad");
  }
  if (dtype == B200_DT_FLOAT) {
    if (p.vec == 4)
      launch_pdl(bias_grad_stage1<float, 4>, dim3(grid), dim3(block), 0, s, static_cast<const float*>(out_backprop),
                                                        partial, rows, (int)channels,
                                                        p.rows_per_chunk, nullptr, nullptr);
    else
      launch_pdl(bias_grad_stage1<float, 1>, dim3(grid), dim3(block), 0, s, static_cast<const float*>(out_backprop),
                                                        partial, rows, (int)channels,
                                                        p.rows_per_chunk, nullptr, nullptr);
    launch_pdl(bias_grad_stage2<float>, dim3((unsigned)((channels + 31) / 32)), dim3(block), 0, s, 
        partial, static_cast<float*>(out), p.nchunks, (int)channels);
  } else {
    if (p.vec == 8)
      launch_pdl(bias_grad_stage1<__nv_bfloat16, 8>, dim3(grid), dim3(block), 0, s, 
          static_cast<const __nv_bfloat16*>(out_backprop), partial, rows, (int)channels,
          p.rows_per_chunk, nullptr, nullptr);
    else
      launch_pdl(bias_grad_stage1<__nv_bfloat16, 1>, dim3(grid), dim3(block), 0, s, 
          static_cast<const __nv_bfloat16*>(out_backprop), partial, rows, (int)channels,
          p.rows_per_chunk, nullptr, nullptr);
    launch_pdl(bias_grad_stage2<__nv_bfloat16>, dim3((unsigned)((channels + 31) / 32)), dim3(block), 0, s, 
        partial, static_cast<__nv_bfloat16*>(out), p.nchunks, (int)channels);
  }
  note_launch(2);
  return check_launch("b200_bias_add_grad");
}

int b200_softmax(int dtype, const void* logits, void* out, int64_t rows, int64_t cols,
                 int log_softmax, void* stream) {
  if (rows < 0 || cols < 0 || cols > INT32_MAX) {
    set_last_error("b200_softmax: bad shape [%lld, %lld]", (long long)rows, (long long)cols);
    return B200_INVALID_ARGUMENT;
  }
  if (rows * cols == 0) return B200_OK;
  int rc = require_device("b200_softmax");
  if (rc) return rc;
  if (dtype == B200_DT_FLOAT)
    return launch_softmax<float>(logits, out, rows, (int)cols, log_softmax != 0, as_stream(stream));
  if (dtype == B200_DT_BFLOAT16)
    return launch_softmax<__nv_bfloat16>(logits, out, rows, (int)cols, log_softmax != 0,
                                         as_stream(stream));
  set_last_error("b200_softmax: unsupported dtype %d", dtype);
  return B200_UNIMPLEMENTED;
}

int b200_softmax_xent(int dtype, const void* logits, const void* labels, void* loss,
                      void* backprop, int64_t rows, int64_t cols, void* stream) {
  return b200_softmax_xent_scaled(dtype, logits, labels, loss, backprop, rows, cols, nullptr, stream);
}

int b200_softmax_xent_scaled(int dtype, const void* logits, const void* labels, void* loss,
                             void* backprop, int64_t rows, int64_t cols,
                             const float* backprop_scale, void* stream) {
  const float* sc = backprop_scale;
  if (sc != nullptr && dtype != B200_DT_FLOAT) {
    set_last_error("b200_softmax_xent_scaled: the fused scale is fp32-only");
    return B200_UNIMPLEMENTED;
  }
  if (rows < 0 || cols < 0 || cols > INT32_MAX) {
    set_last_error("b200_softmax_xent: bad shape [%lld, %lld]", (long long)rows, (long long)cols);
    return B200_INVALID_ARGUMENT;
  }
  if (rows == 0) return B200_OK;
  int rc = require_device("b200_softmax_xent");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
  if (cols == 0) return b200_memset_async(loss, 0, (size_t)rows * (dtype == B200_DT_FLOAT ? 4 : 2), stream);
  if (dtype == B200_DT_FLOAT) {
    const bool vec = cols % 4 == 0 && cols <= 1024 && aligned16(logits) && aligned16(labels) &&
                     aligned16(backprop);
    const float* xl = static_cast<const float*>(logits);
    const float* ll = static_cast<const float*>(labels);
    float* lo = static_cast<float*>(loss);
    float* bo = static_cast<float*>(backprop);
    unsigned wg = (unsigned)((rows + 7) / 8);
    if (wg > 8u * (unsigned)sm_count()) wg = 8u * (unsigned)sm_count();
    if (vec && cols <= 128)
      launch_pdl(xent_warp_vec_kernel<1>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols, sc);
    else if (vec && cols <= 256)
      launch_pdl(xent_warp_vec_kernel<2>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols, sc);
    else if (vec && cols <= 512)
      launch_pdl(xent_warp_vec_kernel<4>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols, sc);
    else if (vec)
      launch_pdl(xent_warp_vec_kernel<8>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols, sc);
    else if (cols <= 1024)
      launch_pdl(xent_warp_kernel<float>, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, s, 
          static_cast<const float*>(logits), static_cast<const float*>(labels),
          static_cast<float*>(loss), static_cast<float*>(backprop), rows, (int)cols, sc);
    else
      launch_pdl(xent_block_kernel<float>, dim3((unsigned)rows), dim3(256), 0, s, 
          static_cast<const float*>(logits), static_cast<const float*>(labels),
          static_cast<float*>(loss), static_cast<float*>(backprop), (int)cols, sc);
  } else if (dtype == B200_DT_BFLOAT16) {
    const bool vec = cols % 8 == 0 && cols <= 1024 && aligned16(logits) && aligned16(labels) &&
                     aligned16(backprop);
    const __nv_bfloat16* xl = static_cast<const __nv_bfloat16*>(logits);
    const __nv_bfloat16* ll = static_cast<const __nv_bfloat16*>(labels);
    __nv_bfloat16* lo = static_cast<__nv_bfloat16*>(loss);
    __nv_bfloat16* bo = static_cast<__nv_bfloat16*>(backprop);
    unsigned wg = (unsigned)((rows + 7) / 8);
    if (wg > 8u * (unsigned)sm_count()) wg = 8u * (unsigned)sm_count();
    if (vec && cols <= 256)
      launch_pdl(xent_warp_vec_bf16_kernel<1>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols);
    else if (vec && cols <= 512)
      launch_pdl(xent_warp_vec_bf16_kernel<2>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols);
    else if (vec)
      launch_pdl(xent_warp_vec_bf16_kernel<4>, dim3(wg), dim3(256), 0, s, xl, ll, lo, bo, rows, (int)cols);
    else if (cols <= 1024)
      launch_pdl(xent_warp_kernel<__nv_bfloat16>, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, s, 
          static_cast<const __nv_bfloat16*>(logits), static_cast<const __nv_bfloat16*>(labels),
          static_cast<__nv_bfloat16*>(loss), static_cast<__nv_bfloat16*>(backprop), rows,
          (int)cols, nullptr);
    else
      launch_pdl(xent_block_kernel<__nv_bfloat16>, dim3((unsigned)rows), dim3(256), 0, s, 
          static_cast<const __nv_bfloat16*>(logits), static_cast<const __nv_bfloat16*>(labels),
          static_cast<__nv_bfloat16*>(loss), static_cast<__nv_bfloat16*>(backprop), (int)cols,
          nullptr);
  } else {
    set_last_error("b200_softmax_xent: unsupported dtype %d", dtype);
    return B200_UNIMPLEMENTED;
  }
  note_launch();
  return check_launch("b200_softmax_xent");
}

int b200_argmax(int dtype, const void* in, int64_t* out, int64_t outer, int64_t axis_size,
                int64_t inner, void* stream) {
  if (outer < 0 || inner < 0 || axis_size <= 0) {
    set_last_error("b200_argmax: bad shape [%lld, %lld, %lld] (axis must be non-empty)",
                   (long long)outer, (long long)axis_size, (long long)inner);
    return B200_INVALID_ARGUMENT;
  }
  if (outer * inner == 0) return B200_OK;
  int rc = require_device("b200_argmax");
  if (rc) return rc;
  cudaStream_t s = as_stream(stream);
#define ARG_LAUNCH(T)                                                                          \
  do {                                                                                         \
    if (inner == 1 && axis_size >= 64)                                                         \
      launch_pdl(argmax_last_axis_kernel<T>, dim3((unsigned)((outer + 7) / 8)), dim3(256), 0, s,                   \
          static_cast<const T*>(in), out, outer, axis_size);                                   \
    else                                                                                       \
      launch_pdl(argmax_strided_kernel<T>, dim3((unsigned)((outer * inner + 255) / 256)), dim3(256), 0, s,         \
          static_cast<const T*>(in), out, outer, axis_size, inner);                            \
  } while (0)
  if (dtype == B200_DT_FLOAT)
    ARG_LAUNCH(float);
  else if (dtype == B200_DT_INT32)
    ARG_LAUNCH(int32_t);
  else if (dtype == B200_DT_INT64)
    ARG_LAUNCH(int64_t);
  else {
    set_last_error("b200_argmax: unsupported dtype %d", dtype);
    return B200_UNIMPLEMENTED;
  }
#undef ARG_LAUNCH
  note_launch();
  return check_launch("b200_argmax");
}

int b200_reduce_sum(int dtype, const void* in, float scale, void* out, int64_t n, void* stream) {
  return b200_reduce(dtype, in, out, 1, n, 1, scale, stream);
}

int b200_reduce(int dtype, const void* in, void* out, int64_t outer, int64_t reduce, int64_t inner,
                float scale, void* stream) {
  if (outer < 0 || reduce < 0 || inner < 0) {
    set_last_error("b200_reduce: negative extent (%lld, %lld, %lld)", (long long)outer,
                   (long long)reduce, (long long)inner);
    return B200_INVALID_ARGUMENT;
  }
  if (dtype != B200_DT_FLOAT && dtype != B200_DT_BFLOAT16) {
    set_last_error("b200_reduce: only DT_FLOAT / DT_BFLOAT16 are supported (got %d)", dtype);
    return B200_UNIMPLEMENTED;
  }
  if (outer == 0 || inner == 0) return B200_OK;  // empty output
  if (outer > 0x7fffffffLL || (inner + 31) / 32 > 0x7fffffffLL) {
    set_last_error("b200_reduce: extent beyond the launch grid (outer %lld, inner %lld)",
                   (long long)outer, (long long)inner);
    return B200_UNIMPLEMENTED;
  }
  int rc = require_device("b200_reduce");
  if (rc) return rc;
  // reduce == 0: the sum over an empty set is 0 (the kernels' loops simply do not run)
  if (dtype == B200_DT_FLOAT)
    launch_reduce<float>(in, out, outer, reduce, inner, scale, as_stream(stream));
  else
    launch_reduce<__nv_bfloat16>(in, out, outer, reduce, inner, scale, as_stream(stream));
  note_launch();
  return check_launch("b200_reduce");
}

}  // extern "C"
