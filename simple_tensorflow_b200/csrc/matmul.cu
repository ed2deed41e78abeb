// MatMul / BatchMatMul entry points of the C ABI, the precision/shape dispatch in front of the
// tcgen05 GEMM, and the SIMT fp32 GEMM that serves shapes TMA cannot address (leading dimension
// not a multiple of 16 bytes, e.g. the 3x5 matrices of the reference's matmul_op_test.py) and
// the "exact fp32" precision mode.
//
// Reference semantics: MatMulOp::Compute (tensorflow/core/kernels/matmul_op.cc:215-256) and
// BatchMatMul::Compute (tensorflow/core/kernels/batch_matmul_op_impl.h:367-434).
#include <cuda_bf16.h>

#include "b200_internal.h"

namespace b200 {

template <typename T>
__device__ __forceinline__ float to_f32(T v);
template <>
__device__ __forceinline__ float to_f32<float>(float v) {
  return v;
}
template <>
__device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) {
  return __bfloat162float(v);
}
template <typename T>
__device__ __forceinline__ T from_f32(float v);
template <>
__device__ __forceinline__ float from_f32<float>(float v) {
  return v;
}
template <>
__device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

// 64x64 output tile, 16x16 threads, 4x4 micro-tile per thread, K step 16.  Any strides/major.
constexpr int kSimtTile = 64;
constexpr int kSimtK = 16;

template <typename T>
__global__ void __launch_bounds__(256)
gemm_simt_kernel(const T* __restrict__ A, const T* __restrict__ B, T* __restrict__ C, int M, int N,
                 int K, long long lda, long long ldb, long long ldc, long long sA, long long sB,
                 long long sC, bool a_mn, bool b_mn) {
  pdl_prologue();
  __shared__ float As[kSimtK][kSimtTile + 1];
  __shared__ float Bs[kSimtK][kSimtTile + 1];
  const int batch = blockIdx.z;
  A += batch * sA;
  B += batch * sB;
  C += batch * sC;
  const int m0 = blockIdx.y * kSimtTile;
  const int n0 = blockIdx.x * kSimtTile;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += kSimtK) {
    // cooperative load: 64x16 elements of A and of B, 4 per thread each
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int idx = threadIdx.x + i * 256;
      int mm, kk;
      if (a_mn) {  // stored [K, M]: contiguous along M
        mm = idx & 63;
        kk = idx >> 6;
      } else {  // stored [M, K]: contiguous along K
        kk = idx & 15;
        mm = idx >> 4;
      }
      const int gm = m0 + mm, gk = k0 + kk;
      float v = 0.f;
      if (gm < M && gk < K) v = to_f32<T>(a_mn ? A[(long long)gk * lda + gm] : A[(long long)gm * lda + gk]);
      As[kk][mm] = v;
      int nn;
      if (b_mn) {  // stored [K, N]
        nn = idx & 63;
        kk = idx >> 6;
      } else {  // stored [N, K]
        kk = idx & 15;
        nn = idx >> 4;
      }
      const int gn = n0 + nn;
      const int gk2 = k0 + kk;
      v = 0.f;
      if (gn < N && gk2 < K) v = to_f32<T>(b_mn ? B[(long long)gk2 * ldb + gn] : B[(long long)gn * ldb + gk2]);
      Bs[kk][nn] = v;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kSimtK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gm = m0 + ty * 4 + i;
    if (gm >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int gn = n0 + tx * 4 + j;
      if (gn < N) C[(long long)gm * ldc + gn] = from_f32<T>(acc[i][j]);
    }
  }
}

// Skinny GEMM for N <= 32 (the 10-class logits layer, its weight gradient): the problem is a few MB
// and a few MFLOP, so what matters is how many independent loads are in flight, not FLOPs.  Two
// thread maps, both with the K range of a row split over several warps of the CTA, four k steps
// unrolled (independent loads) and a fixed-order merge through shared memory (reproducible):
//   A stored [M, K] (K contiguous):  lanes stride over k (coalesced), 2 rows x 4 K-splits per CTA,
//                                    lanes folded by shuffles;
//   A stored [K, M] (M contiguous):  lanes are 32 consecutive rows (coalesced), 8 K-splits per CTA,
//                                    B[k, :] is the same address for the whole warp (broadcast).
// The 64x64-tile kernel above would put such a problem on a handful of CTAs.
template <typename T, int NMAX>
__global__ void __launch_bounds__(256)
gemm_skinny_kernel(const T* __restrict__ A, const T* __restrict__ B, T* __restrict__ C, int M, int N,
                   int K, long long lda, long long ldb, long long ldc, bool a_mn, bool b_mn,
                   long long strideA, long long strideB, long long strideC, bool c_t) {
  pdl_prologue();
  // batch = blockIdx.y.  c_t: C is written transposed (element (row, j) at C[j * ldc + row]) --
  // how a skinny-M product runs here as its transpose (C^T = B^T A^T).
  A += (long long)blockIdx.y * strideA;
  B += (long long)blockIdx.y * strideB;
  C += (long long)blockIdx.y * strideC;
  // B is staged per K chunk as Bs[k][NMAX (+4 pad)] fp32, zero filled past N / K: the inner loops
  // are 16-byte shared loads (broadcast, or conflict-free thanks to the pad) and plain FMAs, with
  // no layout or bounds predicate left in them.
  constexpr int KC = NMAX <= 16 ? 512 : 256;
  constexpr int LDB = NMAX + 4;
  constexpr int kRed = 8 * NMAX * 33;
  __shared__ __align__(16) float sm[KC * LDB > kRed ? KC * LDB : kRed];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float acc[NMAX];
#pragma unroll
  for (int j = 0; j < NMAX; ++j) acc[j] = 0.f;
  const int wr = warp >> 2, wq = warp & 3;  // K-major A: 2 rows x 4 K-splits
  const int row = a_mn ? blockIdx.x * 32 + lane : blockIdx.x * 2 + wr;
  const bool ok = row < M;
  for (int kc = 0; kc < K; kc += KC) {
    __syncthreads();  // the previous chunk's readers are done
    for (int i = threadIdx.x; i < KC * NMAX; i += 256) {
      const int k = b_mn ? i / NMAX : i % KC, j = b_mn ? i % NMAX : i / KC;
      float v = 0.f;
      if (kc + k < K && j < N)
        v = to_f32<T>(b_mn ? B[(long long)(kc + k) * ldb + j] : B[(long long)j * ldb + kc + k]);
      sm[k * LDB + j] = v;
    }
    __syncthreads();
    if (!a_mn) {
      // lane owns k = kc + wq * (KC / 4) + lane + 32 u: coalesced, KC / 128 loads in flight
      constexpr int U = KC / 128;
      const int kb = wq * (KC / 4) + lane;
      float a[U];
#pragma unroll
      for (int u = 0; u < U; ++u)
        a[u] = ok && kc + kb + 32 * u < K ? to_f32<T>(A[(long long)row * lda + kc + kb + 32 * u]) : 0.f;
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float4* bp = reinterpret_cast<const float4*>(sm + (kb + 32 * u) * LDB);
#pragma unroll
        for (int q = 0; q < NMAX / 4; ++q) {
          const float4 bv = bp[q];
          acc[4 * q] = fmaf(a[u], bv.x, acc[4 * q]);
          acc[4 * q + 1] = fmaf(a[u], bv.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(a[u], bv.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(a[u], bv.w, acc[4 * q + 3]);
        }
      }
    } else {
      // lane = row (coalesced along M), warp w owns k = kc + w + 8 i; 8 A loads in flight
      constexpr int U = 8;
      for (int k0 = warp; k0 < KC; k0 += 8 * U) {
        float a[U];
#pragma unroll
        for (int u = 0; u < U; ++u)
          a[u] = ok && kc + k0 + 8 * u < K ? to_f32<T>(A[(long long)(kc + k0 + 8 * u) * lda + row]) : 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const float4* bp = reinterpret_cast<const float4*>(sm + (k0 + 8 * u) * LDB);
#pragma unroll
          for (int q = 0; q < NMAX / 4; ++q) {
            const float4 bv = bp[q];
            acc[4 * q] = fmaf(a[u], bv.x, acc[4 * q]);
            acc[4 * q + 1] = fmaf(a[u], bv.y, acc[4 * q + 1]);
            acc[4 * q + 2] = fmaf(a[u], bv.z, acc[4 * q + 2]);
            acc[4 * q + 3] = fmaf(a[u], bv.w, acc[4 * q + 3]);
          }
        }
      }
    }
  }
  __syncthreads();  // Bs is dead: the merge buffer red[8][NMAX][33] lives in the same bytes
  float* red = sm;
  if (!a_mn) {
#pragma unroll
    for (int j = 0; j < NMAX; ++j) {
      float v = acc[j];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if (lane == 0) red[(warp * NMAX + j) * 33] = v;
    }
    __syncthreads();
    if (threadIdx.x < 2 * NMAX) {
      const int r = threadIdx.x / NMAX, j = threadIdx.x % NMAX;
      const int orow = blockIdx.x * 2 + r;
      if (orow < M && j < N) {
        float v = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) v += red[((r * 4 + q) * NMAX + j) * 33];
        C[c_t ? (long long)j * ldc + orow : (long long)orow * ldc + j] = from_f32<T>(v);
      }
    }
  } else {
#pragma unroll
    for (int j = 0; j < NMAX; ++j) red[(warp * NMAX + j) * 33 + lane] = acc[j];
    __syncthreads();
    for (int i = threadIdx.x; i < 32 * NMAX; i += 256) {
      // consecutive threads -> consecutive C elements in either orientation
      const int r = c_t ? i % 32 : i / NMAX, j = c_t ? i / 32 : i % NMAX;
      const int orow = blockIdx.x * 32 + r;
      if (orow < M && j < N) {
        float v = 0.f;
#pragma unroll
        for (int q = 0; q < 8; ++q) v += red[(q * NMAX + j) * 33 + r];
        C[c_t ? (long long)j * ldc + orow : (long long)orow * ldc + j] = from_f32<T>(v);
      }
    }
  }
}

// Matrix-vector products (N <= 4; vector-matrix ones run transposed): pure bandwidth, no staging.
//   A stored [M, K]: one warp per row, lanes stride over K (coalesced), shuffle fold;
//   A stored [K, M]: one thread per row (a warp reads 32 consecutive rows of every k), B[k, :] is a
//                    broadcast load; eight k in flight.
// Rows are grid-strided; blockIdx.y is the batch.  Fixed summation order (reproducible).
template <typename T, int NV>
__global__ void __launch_bounds__(256)
gemv_kernel(const T* __restrict__ A, const T* __restrict__ B, T* __restrict__ C, int M, int N, int K,
            long long lda, long long ldb, long long ldc, bool a_mn, bool b_mn, long long strideA,
            long long strideB, long long strideC, bool c_t) {
  pdl_prologue();
  A += (long long)blockIdx.y * strideA;
  B += (long long)blockIdx.y * strideB;
  C += (long long)blockIdx.y * strideC;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  auto bval = [&](int k, int j) {
    return to_f32<T>(b_mn ? B[(long long)k * ldb + j] : B[(long long)j * ldb + k]);
  };
  if (!a_mn) {
    for (long long row = (long long)blockIdx.x * 8 + warp; row < M; row += (long long)gridDim.x * 8) {
      const T* arow = A + row * lda;
      float acc[NV];
#pragma unroll
      for (int j = 0; j < NV; ++j) acc[j] = 0.f;
      constexpr int U = 8;
      for (int k0 = lane; k0 < K; k0 += 32 * U) {
        float a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) a[u] = k0 + 32 * u < K ? to_f32<T>(arow[k0 + 32 * u]) : 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (k0 + 32 * u < K) {
#pragma unroll
            for (int j = 0; j < NV; ++j)
              if (j < N) acc[j] = fmaf(a[u], bval(k0 + 32 * u, j), acc[j]);
          }
      }
#pragma unroll
      for (int j = 0; j < NV; ++j) {
        float v = acc[j];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0 && j < N)
          C[c_t ? (long long)j * ldc + row : row * ldc + j] = from_f32<T>(v);
      }
    }
  } else {
    for (long long row = (long long)blockIdx.x * 256 + threadIdx.x; row < M;
         row += (long long)gridDim.x * 256) {
      float acc[NV];
#pragma unroll
      for (int j = 0; j < NV; ++j) acc[j] = 0.f;
      constexpr int U = 8;
      for (int k0 = 0; k0 < K; k0 += U) {
        float a[U];
#pragma unroll
        for (int u = 0; u < U; ++u) a[u] = k0 + u < K ? to_f32<T>(A[(long long)(k0 + u) * lda + row]) : 0.f;
#pragma unroll
        for (int u = 0; u < U; ++u)
          if (k0 + u < K) {
#pragma unroll
            for (int j = 0; j < NV; ++j)
              if (j < N) acc[j] = fmaf(a[u], bval(k0 + u, j), acc[j]);
          }
      }
#pragma unroll
      for (int j = 0; j < NV; ++j)
        if (j < N) C[c_t ? (long long)j * ldc + row : row * ldc + j] = from_f32<T>(acc[j]);
    }
  }
}

int gemm_simt(const GemmArgs& g, cudaStream_t stream) {
  // N <= 4 / M <= 4: matrix-vector and vector-matrix products (batch_matmul_op_test.cc:107-132);
  // N <= 32: the skinny kernel (the 10-class layer).  A skinny-M problem runs as its transpose
  // C^T[N, M] = B^T[N, K] A^T[K, M].
  const bool gemv_n = g.N <= 4 && g.M >= 64;
  const bool gemv_m = !gemv_n && g.M <= 4 && g.N >= 64;
  const bool skinny_n = !gemv_n && !gemv_m && g.batch == 1 && g.N <= 32 && g.K >= 64 && g.M >= 64;
  if ((gemv_n || gemv_m || skinny_n) && g.batch <= 65535) {
    const void *pa = g.a, *pb = g.b;
    long long M = g.M, N = g.N, lda = g.lda, ldb = g.ldb, sA = g.strideA, sB = g.strideB;
    bool a_mn = g.a_mn_major, b_mn = g.b_mn_major;
    if (gemv_m) {  // A' = B^T (stored as B), B' = A^T (stored as A)
      pa = g.b; pb = g.a;
      M = g.N; N = g.M;
      lda = g.ldb; ldb = g.lda;
      sA = g.strideB; sB = g.strideA;
      a_mn = g.b_mn_major;   // B stored [K, N] = A' stored [K, M']
      b_mn = g.a_mn_major;   // A stored [K, M] = B' stored [K, N']
    }
    if (gemv_n || gemv_m) {
      const long long units = a_mn ? (M + 255) / 256 : (M + 7) / 8;
      const long long cap = std::max<long long>(1, 16LL * sm_count() / g.batch);
      const dim3 grid((unsigned)std::min(units, cap), (unsigned)g.batch);
#define GEMV(T)                                                                                   \
  launch_pdl(gemv_kernel<T, 4>, grid, dim3(256), 0, stream, static_cast<const T*>(pa),            \
             static_cast<const T*>(pb), static_cast<T*>(g.c), (int)M, (int)N, (int)g.K, lda, ldb, \
             g.ldc, a_mn, b_mn, sA, sB, g.strideC, gemv_m)
      if (g.dtype == B200_DT_FLOAT) {
        GEMV(float);
      } else if (g.dtype == B200_DT_BFLOAT16) {
        GEMV(__nv_bfloat16);
      } else {
        set_last_error("gemm_simt: unsupported dtype %d", g.dtype);
        return B200_UNIMPLEMENTED;
      }
#undef GEMV
      note_launch();
      return check_launch("gemv");
    }
    const dim3 grid(a_mn ? (unsigned)((M + 31) / 32) : (unsigned)((M + 1) / 2), 1);
#define SKINNY(T, NMAX)                                                                          \
  launch_pdl(gemm_skinny_kernel<T, NMAX>, grid, dim3(256), 0, stream, static_cast<const T*>(pa), \
             static_cast<const T*>(pb), static_cast<T*>(g.c), (int)M, (int)N, (int)g.K, lda,     \
             ldb, g.ldc, a_mn, b_mn, sA, sB, g.strideC, false)
    if (g.dtype == B200_DT_FLOAT) {
      if (N <= 16) SKINNY(float, 16); else SKINNY(float, 32);
    } else if (g.dtype == B200_DT_BFLOAT16) {
      if (N <= 16) SKINNY(__nv_bfloat16, 16); else SKINNY(__nv_bfloat16, 32);
    } else {
      set_last_error("gemm_simt: unsupported dtype %d", g.dtype);
      return B200_UNIMPLEMENTED;
    }
#undef SKINNY
    note_launch();
    return check_launch("gemm_skinny");
  }
  if (g.batch > 65535) {
    set_last_error("gemm_simt: batch %lld exceeds grid.z limit", g.batch);
    return B200_UNIMPLEMENTED;
  }
  dim3 grid((unsigned)((g.N + kSimtTile - 1) / kSimtTile),
            (unsigned)((g.M + kSimtTile - 1) / kSimtTile), (unsigned)g.batch);
  if (g.dtype == B200_DT_FLOAT) {
    launch_pdl(gemm_simt_kernel<float>, dim3(grid), dim3(256), 0, stream, 
        static_cast<const float*>(g.a), static_cast<const float*>(g.b), static_cast<float*>(g.c),
        (int)g.M, (int)g.N, (int)g.K, g.lda, g.ldb, g.ldc, g.strideA, g.strideB, g.strideC,
        g.a_mn_major, g.b_mn_major);
  } else if (g.dtype == B200_DT_BFLOAT16) {
    launch_pdl(gemm_simt_kernel<__nv_bfloat16>, dim3(grid), dim3(256), 0, stream, 
        static_cast<const __nv_bfloat16*>(g.a), static_cast<const __nv_bfloat16*>(g.b),
        static_cast<__nv_bfloat16*>(g.c), (int)g.M, (int)g.N, (int)g.K, g.lda, g.ldb, g.ldc,
        g.strideA, g.strideB, g.strideC, g.a_mn_major, g.b_mn_major);
  } else {
    set_last_error("gemm_simt: unsupported dtype %d", g.dtype);
    return B200_UNIMPLEMENTED;
  }
  note_launch();
  return check_launch("gemm_simt");
}

// Tensor-core or CUDA-core kernel for this problem.  MatMul and the fused MatMul both ask here, so
// adding a BiasAdd / Relu / ReluGrad tail never changes which kernel (and which arithmetic, TF32 or
// IEEE fp32) computes the product.
static bool use_tcgen05(const GemmArgs& g) {
  const bool want_exact = g.dtype == B200_DT_FLOAT && b200_get_matmul_precision() == 1;
  // Tiny problems: a 128-row MMA tile would be mostly padding and launch-bound anyway.
  const bool tiny = g.M * g.N * g.K < 32LL * 32 * 32;
  // matrix-vector / vector-matrix products: a 128-row MMA tile would be > 96 % padding; they are
  // bandwidth problems for the K-split CUDA-core kernel (exact fp32)
  const bool gemv_like = (g.N <= 4 && g.M >= 64) || (g.M <= 4 && g.N >= 64);
  return !want_exact && !tiny && !gemv_like && gemm_tcgen05_supported(g) &&
         driver().cuTensorMapEncodeTiled;
}

int gemm_dispatch(const GemmArgs& g, cudaStream_t stream) {
  return use_tcgen05(g) ? gemm_tcgen05(g, stream) : gemm_simt(g, stream);
}

static int validate_gemm(const char* what, int dtype, const void* a, const void* b, void* c,
                         int64_t m, int64_t n, int64_t k, int64_t batch) {
  if (dtype != B200_DT_FLOAT && dtype != B200_DT_BFLOAT16) {
    set_last_error("%s: unsupported dtype %d (DT_FLOAT=1, DT_BFLOAT16=14)", what, dtype);
    return B200_UNIMPLEMENTED;
  }
  if (m <= 0 || n <= 0 || k <= 0 || batch <= 0) {
    set_last_error("%s: m, n, k, batch must be positive (m=%lld n=%lld k=%lld batch=%lld); the "
                   "zero-size rules of matmul_op.cc:240-253 belong to the OpKernel wrapper",
                   what, (long long)m, (long long)n, (long long)k, (long long)batch);
    return B200_INVALID_ARGUMENT;
  }
  if (!a || !b || !c) {
    set_last_error("%s: null pointer argument", what);
    return B200_INVALID_ARGUMENT;
  }
  if (m > INT32_MAX || n > INT32_MAX || k > INT32_MAX) {
    set_last_error("%s: dimension exceeds int32", what);
    return B200_INVALID_ARGUMENT;
  }
  return require_device(what);
}

// Arguments of one row-major product C[batch][m, n] = op(A) * op(B), validated under the name
// `what`: an optional fused tail (bias, relu or relu-grad features) and optional scratch that lets
// the product split K.
static int product_args(const char* what, int dtype, const void* a, const void* b, void* c,
                        int64_t batch, int64_t m, int64_t n, int64_t k, int transpose_a,
                        int transpose_b, const void* bias, int relu,
                        const void* relu_grad_features, void* workspace, size_t workspace_bytes,
                        GemmArgs* out) {
  int rc = validate_gemm(what, dtype, a, b, c, m, n, k, batch);
  if (rc) return rc;
  if (relu && relu_grad_features) {
    set_last_error("%s: relu and relu_grad_features are mutually exclusive", what);
    return B200_INVALID_ARGUMENT;
  }
  GemmArgs g{};
  g.dtype = dtype;
  g.a = a;
  g.b = b;
  g.c = c;
  g.M = m;
  g.N = n;
  g.K = k;
  g.batch = batch;
  g.lda = transpose_a ? m : k;
  g.ldb = transpose_b ? k : n;
  g.ldc = n;
  g.strideA = m * k;
  g.strideB = k * n;
  g.strideC = m * n;
  g.a_mn_major = transpose_a != 0;
  g.b_mn_major = transpose_b == 0;
  g.bias = bias;
  g.relu = relu != 0;
  g.relu_grad_features = relu_grad_features;
  g.ld_features = n;
  if (workspace != nullptr && workspace_bytes > 0 && relu_grad_features == nullptr) {
    g.workspace = workspace;  // enables split-K; the bias / relu tail moves to the reduction pass
    g.workspace_bytes = workspace_bytes;
  }
  *out = g;
  return B200_OK;
}

static int fused_matmul(const GemmArgs& g, cudaStream_t stream) {
  if (use_tcgen05(g)) return gemm_tcgen05(g, stream);
  // CUDA-core shapes (TMA cannot address them, tiny, matrix-vector) and exact mode: GEMM, then the
  // element-wise tail as separate kernels.
  int rc = gemm_simt(g, stream);
  if (rc) return rc;
  void* c = g.c;
  if (g.bias) rc = b200_bias_add(g.dtype, c, g.bias, c, g.M, g.N, stream);
  if (!rc && g.relu) rc = b200_relu(g.dtype, c, c, g.M * g.N, stream);
  if (!rc && g.relu_grad_features)
    rc = b200_relu_grad(g.dtype, c, g.relu_grad_features, c, g.M * g.N, stream);
  return rc;
}

static size_t align256(size_t x) { return (x + 255) & ~static_cast<size_t>(255); }

}  // namespace b200

using namespace b200;

extern "C" {

size_t b200_matmul_workspace_bytes(int dtype, int64_t m, int64_t n, int64_t k) {
  return gemm_workspace_bytes(dtype, m, n, k, 1);
}

int b200_matmul(int dtype, const void* a, const void* b, void* c, int64_t m, int64_t n, int64_t k,
                int transpose_a, int transpose_b, void* workspace, size_t workspace_bytes,
                void* stream) {
  GemmArgs g;
  const int rc = product_args("b200_matmul", dtype, a, b, c, 1, m, n, k, transpose_a, transpose_b,
                              nullptr, 0, nullptr, workspace, workspace_bytes, &g);
  return rc ? rc : fused_matmul(g, as_stream(stream));
}

int b200_fused_matmul(int dtype, const void* a, const void* b, void* c, int64_t m, int64_t n,
                      int64_t k, int transpose_a, int transpose_b, const void* bias, int relu,
                      const void* relu_grad_features, void* stream) {
  return b200_fused_matmul_ws(dtype, a, b, c, m, n, k, transpose_a, transpose_b, bias, relu,
                              relu_grad_features, nullptr, 0, stream);
}

int b200_fused_matmul_ws(int dtype, const void* a, const void* b, void* c, int64_t m, int64_t n,
                         int64_t k, int transpose_a, int transpose_b, const void* bias, int relu,
                         const void* relu_grad_features, void* workspace, size_t workspace_bytes,
                         void* stream) {
  GemmArgs g;
  const int rc = product_args("b200_fused_matmul", dtype, a, b, c, 1, m, n, k, transpose_a,
                              transpose_b, bias, relu, relu_grad_features, workspace,
                              workspace_bytes, &g);
  return rc ? rc : fused_matmul(g, as_stream(stream));
}

size_t b200_matmul_pair_workspace_bytes(int dtype, int64_t m0, int64_t n0, int64_t k0, int64_t m1,
                                        int64_t n1, int64_t k1) {
  const size_t ws1 = gemm_workspace_bytes(dtype, m1, n1, k1, 1);
  return ws1 ? align256(gemm_workspace_bytes(dtype, m0, n0, k0, 1)) + ws1
             : gemm_workspace_bytes(dtype, m0, n0, k0, 1);
}

int b200_matmul_pair(int dtype, const void* a0, const void* b0, void* c0, int64_t m0, int64_t n0,
                     int64_t k0, int transpose_a0, int transpose_b0, const void* bias0, int relu0,
                     const void* relu_grad_features0, const void* a1, const void* b1, void* c1,
                     int64_t m1, int64_t n1, int64_t k1, int transpose_a1, int transpose_b1,
                     const void* bias1, int relu1, const void* relu_grad_features1,
                     void* workspace, size_t workspace_bytes, void* stream) {
  // product 0's scratch at offset 0, product 1's at the next 256-byte boundary past it
  const size_t ws0 = workspace ? gemm_workspace_bytes(dtype, m0, n0, k0, 1) : 0;
  const size_t off1 = align256(ws0);
  void* w1 = workspace_bytes > off1 ? static_cast<char*>(workspace) + off1 : nullptr;
  GemmArgs g0, g1;
  int rc = product_args("b200_matmul_pair", dtype, a0, b0, c0, 1, m0, n0, k0, transpose_a0,
                        transpose_b0, bias0, relu0, relu_grad_features0, workspace,
                        std::min(ws0, workspace_bytes), &g0);
  if (rc) return rc;
  rc = product_args("b200_matmul_pair", dtype, a1, b1, c1, 1, m1, n1, k1, transpose_a1,
                    transpose_b1, bias1, relu1, relu_grad_features1, w1,
                    w1 ? workspace_bytes - off1 : 0, &g1);
  if (rc) return rc;
  const cudaStream_t s = as_stream(stream);
  if (use_tcgen05(g0) && use_tcgen05(g1)) return gemm_tcgen05_pair(g0, g1, s);
  rc = fused_matmul(g0, s);
  return rc ? rc : fused_matmul(g1, s);
}

int b200_batch_matmul(int dtype, const void* x, const void* y, void* out, int64_t batch, int64_t m,
                      int64_t n, int64_t k, int adj_x, int adj_y, void* stream) {
  GemmArgs g;
  const int rc = product_args("b200_batch_matmul", dtype, x, y, out, batch, m, n, k, adj_x, adj_y,
                              nullptr, 0, nullptr, nullptr, 0, &g);
  return rc ? rc : gemm_dispatch(g, as_stream(stream));
}

}  // extern "C"
