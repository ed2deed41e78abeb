// Internal (non-ABI) declarations shared by the .cu translation units of libb200tf.so.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b200_ops.h"

namespace b200 {

// printf-style; stores a thread-local message returned by b200_last_error().
void set_last_error(const char* fmt, ...) __attribute__((format(printf, 1, 2)));

// Driver entry points resolved at run time through cudaGetDriverEntryPoint so that the library
// loads (and exports its symbols) on a machine without libcuda.so.
struct DriverApi {
  CUresult (*cuTensorMapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                     const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                     const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                     CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  CUresult (*cuTensorMapEncodeIm2col)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                      const cuuint64_t*, const cuuint64_t*, const int*, const int*,
                                      cuuint32_t, cuuint32_t, const cuuint32_t*,
                                      CUtensorMapInterleave, CUtensorMapSwizzle,
                                      CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
};
const DriverApi& driver();

int sm_count();                       // SMs of the current device (cached per device)
void note_launch(int n = 1);          // bump the library-wide launch counter
int check_launch(const char* what);   // cudaGetLastError -> B200_INTERNAL + message
int require_device(const char* what); // B200_INTERNAL when no CUDA device is usable

inline cudaStream_t as_stream(void* s) { return static_cast<cudaStream_t>(s); }

// ------------------------------------------------------------------ GEMM plumbing
// Implicit-GEMM convolution: the A operand [N*OH*OW, R*S*C] is never materialised; the GEMM's TMA
// producer gathers it from the NHWC activation tensor with im2col-mode loads.
struct ConvAOperand {
  const void* input;  // NHWC
  int N, H, W, C, R, S, OH, OW, sh, sw, pt, pl;
};
struct GemmArgs {
  int dtype;                 // B200_DT_FLOAT or B200_DT_BFLOAT16
  const void* a;             // logical A[M,K]
  const void* b;             // logical B[K,N]
  void* c;                   // C[M,N] row-major
  long long M, N, K, batch;
  long long lda, ldb, ldc;   // leading dimensions of the STORED row-major matrices (elements)
  long long strideA, strideB, strideC;  // batch strides (elements)
  bool a_mn_major;           // A stored as [K,M] (transpose_a)
  bool b_mn_major;           // B stored as [K,N] (i.e. NOT transpose_b)
  void* workspace;           // optional device scratch enabling split-K (may be null)
  size_t workspace_bytes;
  // fused epilogue (tcgen05 path only; all optional)
  const void* bias;                // + bias[col]
  bool relu;                       // max(x, 0)
  const void* relu_grad_features;  // x * (features[row, col] > 0), features [M, N]
  long long ld_features;
  const ConvAOperand* conv_a;      // non-null: A is gathered on the fly (a / lda unused)
};
// Halo-tile implicit-GEMM convolution (conv_halo.cu): unit stride, C and K whole 128-byte channel
// blocks.  `filter` is the row-major [R*S*C, K] matrix (HWIO as stored).
struct ConvHaloArgs {
  const void* input;   // NHWC [N, H, W, C]
  const void* filter;  // [R*S*C, K]
  void* output;        // NHWC [N, OH, OW, K]
  const void* bias;    // optional fused + bias[k]
  bool relu;           // optional fused max(x, 0)
  int N, H, W, C, K, R, S, pt, pl, OH, OW;
};
bool conv_halo_supported(int dtype, const ConvHaloArgs& a);
int conv_halo(int dtype, const ConvHaloArgs& a, cudaStream_t stream);
// Filter gradient on the same idea (conv_halo_wgrad.cu).  ConvHaloArgs here: input = x,
// filter = out_backprop [N, OH, OW, K], output = dW [R*S*C, K]; workspace holds one fp32 partial
// filter gradient per CTA.
bool conv_halo_wgrad_supported(int dtype, const ConvHaloArgs& a);
size_t conv_halo_wgrad_workspace_bytes(int dtype, const ConvHaloArgs& a);
int conv_halo_wgrad(int dtype, const ConvHaloArgs& a, void* workspace, size_t workspace_bytes,
                    cudaStream_t stream);
bool gemm_tcgen05_supported(const GemmArgs& g);
// Can this convolution's patch operand be fetched by TMA im2col (channel / padding limits)?
bool conv_a_supported(int dtype, const ConvAOperand& c);
int gemm_tcgen05(const GemmArgs& g, cudaStream_t stream);
// Two independent tensor-core GEMMs of one dtype (both gemm_tcgen05-eligible) in one persistent
// launch when they share a tile config and their majorness pair is instantiated (one K-major x
// K-major, one MN-major x MN-major: a dense layer's dX and dW); otherwise gemm_tcgen05(a) then
// gemm_tcgen05(b).  Results are bit-identical to the two separate launches.
int gemm_tcgen05_pair(const GemmArgs& a, const GemmArgs& b, cudaStream_t stream);
int gemm_simt(const GemmArgs& g, cudaStream_t stream);
// Precision-aware front door used by matmul / batch_matmul / conv.
int gemm_dispatch(const GemmArgs& g, cudaStream_t stream);
// Optional per-launch timing of the tensor-core GEMM (b200_profile_begin/end): brackets the
// launch with CUDA events on the launching stream.
bool profile_enabled();
void profile_gemm_launch_begin(cudaStream_t stream);
void profile_gemm_launch_end(cudaStream_t stream, double flops);
// Scratch that lets gemm_dispatch use split-K for this shape (0 when it would not split).
size_t gemm_workspace_bytes(int dtype, long long M, long long N, long long K, long long batch);

#ifdef __CUDACC__
// Programmatic dependent launch (sm_90+).  Every kernel of the library executes the trigger first
// thing, so a kernel launched behind it WITH cudaLaunchAttributeProgrammaticStreamSerialization
// (only the tcgen05 GEMM and its split-K reduce) may have its CTAs scheduled while this grid is
// still draining: launch latency and prologue (barrier init, TMEM allocation, cluster sync)
// disappear under the predecessor's tail.  Such a kernel must execute pdl_wait() -- which
// returns once every prerequisite grid has completed and its memory is visible -- before it
// touches global memory.  Both are no-ops for ordinary launches.
__device__ __forceinline__ void pdl_launch_dependents() {
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
// First statement of every kernel but the GEMM (which overlaps its prologue first): let the
// successor be scheduled, then wait for the predecessors' memory.
__device__ __forceinline__ void pdl_prologue() {
  pdl_launch_dependents();
  pdl_wait();
}
void note_collective(bool peer);  // runtime.cu: b200_collective_counts()
bool pdl_enabled();  // runtime.cu: on unless B200TF_NO_PDL is set
// B200TF_KERNEL_TIMES=1 (measurement aid, runtime.cu): every launch is bracketed by CUDA events on
// its stream and the per-kernel totals are printed to stderr at exit (warm caches, in stream
// order; the brackets serialise the launches, so PDL overlap and CUDA graphs are off in this mode).
bool kernel_times_enabled();
void* kernel_times_begin(cudaStream_t stream);
void kernel_times_end(void* token, cudaStream_t stream, const void* kernel);
// kernel<<<grid, block, smem, stream>>>(args...) with programmatic stream serialization allowed:
// the grid may be scheduled while its predecessor in the stream drains (every kernel begins with
// pdl_prologue(), so nothing is read or written before the predecessor has completed).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem,
                              cudaStream_t stream, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  if (kernel_times_enabled()) {
    cfg.numAttrs = 0;
    void* tok = kernel_times_begin(stream);
    const cudaError_t e = cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
    kernel_times_end(tok, stream, reinterpret_cast<const void*>(kernel));
    return e;
  }
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
#endif

}  // namespace b200
