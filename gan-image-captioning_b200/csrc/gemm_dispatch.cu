// GEMM dispatch: tcgen05 tensor-core kernels when the mode and the operand layout allow it,
// the exact-fp32 CUDA-core kernel otherwise.  Both are this library's own kernels; nothing here
// falls back to a CPU or to a vendor library.
#include <stdlib.h>

#include <vector>

#include "gic_internal.cuh"

namespace gic {

struct ProfRec { int kind; double work; cudaEvent_t a, b; };
static bool g_prof = false;
static std::vector<ProfRec> g_recs;
bool prof_enabled() { return g_prof; }
void prof_open(int kind, double work, cudaStream_t s) {
  ProfRec r; r.kind = kind; r.work = work;
  cudaEventCreate(&r.a); cudaEventCreate(&r.b);
  cudaEventRecord(r.a, s);
  g_recs.push_back(r);
}
void prof_close(cudaStream_t s) { if (!g_recs.empty()) cudaEventRecord(g_recs.back().b, s); }
void prof_begin() { g_prof = true; }
// call after the stream has been synchronised
void prof_end(double* ms, double* work, unsigned long long* calls) {
  g_prof = false;
  for (int k = 0; k < PROF_KINDS; ++k) { ms[k] = 0; work[k] = 0; calls[k] = 0; }
  for (auto& r : g_recs) {
    float t = 0.f;
    if (cudaEventElapsedTime(&t, r.a, r.b) == cudaSuccess) { ms[r.kind] += t; work[r.kind] += r.work; calls[r.kind] += 1; }
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  g_recs.clear();
}

int gemm_tc(int mode, bool transA, bool transB, int M, int N, int K, float alpha, const float* A, int lda,
            const float* B, int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream,
            bool* handled);

int gemm_tc_persistent(bool transA, bool transB, int M, int N, int K, float alpha, const float* A, int lda,
                       const float* B, int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream,
                       bool* handled);

int gemm_tc_bf16(bool transA, bool transB, int M, int N, int K, float alpha, const void* A, int lda, const void* B,
                 int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream, bool* handled);

int gemm_bf16(bool transA, bool transB, int M, int N, int K, float alpha, const void* A, int lda, const void* B, int ldb,
              float beta, float* C, int ldc, const float* bias, cudaStream_t stream, int prof_kind) {
  ProfScope prof(prof_kind, 2.0 * M * N * K, stream);
  bool handled = false;
  GIC_TRY(gemm_tc_bf16(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, stream, &handled));
  GIC_REQUIRE(handled, GIC_ERR_UNSUPPORTED, "gemm_bf16: operands must be 16-byte aligned with leading dimensions %% 8 == 0");
  return GIC_OK;
}

__global__ void f32_to_bf16_kernel(const float* __restrict__ src, int rows, int cols, int ld_src,
                                   unsigned short* __restrict__ dst, int ld_dst) {
  const size_t n = (size_t)rows * cols;
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const int r = (int)(i / cols), c = (int)(i % cols);
    const float x = src[(size_t)r * ld_src + c];
    unsigned int u = __float_as_uint(x);
    u += 0x7fffu + ((u >> 16) & 1u);                 // round to nearest even (inputs are finite)
    dst[(size_t)r * ld_dst + c] = (unsigned short)(u >> 16);
  }
}
// four elements per thread: one 16-byte load, one 8-byte store, 32-bit index arithmetic (the scalar kernel spent most of its
// 10 us per call in a 64-bit division per element); same rounding
__global__ void f32_to_bf16_vec_kernel(const float* __restrict__ src, int rows, int cols4, int ld_src,
                                       unsigned short* __restrict__ dst, int ld_dst) {
  const unsigned int n = (unsigned int)rows * (unsigned int)cols4;
  for (unsigned int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const unsigned int r = i / (unsigned int)cols4, c = (i - r * (unsigned int)cols4) * 4u;
    const float4 x = *reinterpret_cast<const float4*>(src + (size_t)r * ld_src + c);
    unsigned int u[4] = {__float_as_uint(x.x), __float_as_uint(x.y), __float_as_uint(x.z), __float_as_uint(x.w)};
#pragma unroll
    for (int e = 0; e < 4; ++e) u[e] = (u[e] + 0x7fffu + ((u[e] >> 16) & 1u)) >> 16;   // round to nearest even (inputs are finite)
    *reinterpret_cast<uint2*>(dst + (size_t)r * ld_dst + c) = make_uint2(u[0] | (u[1] << 16), u[2] | (u[3] << 16));
  }
}
int f32_to_bf16(const float* src, int rows, int cols, int ld_src, void* dst, int ld_dst, cudaStream_t stream) {
  if (rows <= 0 || cols <= 0) return GIC_OK;
  if ((cols % 4) == 0 && (ld_src % 4) == 0 && (ld_dst % 4) == 0 && aligned16(src) && (reinterpret_cast<uintptr_t>(dst) & 7u) == 0 &&
      (long long)rows * (cols / 4) < (1ll << 31)) {
    const int grid = min(cdiv((long long)rows * (cols / 4), 256), 8 * num_sms());
    f32_to_bf16_vec_kernel<<<grid, 256, 0, stream>>>(src, rows, cols / 4, ld_src, reinterpret_cast<unsigned short*>(dst), ld_dst);
    return check_launch("f32_to_bf16_kernel");
  }
  const int grid = min(cdiv((long long)rows * cols, 256), 8 * num_sms());
  f32_to_bf16_kernel<<<grid, 256, 0, stream>>>(src, rows, cols, ld_src, reinterpret_cast<unsigned short*>(dst), ld_dst);
  return check_launch("f32_to_bf16_kernel");
}

int gemm(int mode, bool transA, bool transB, int M, int N, int K, float alpha, const float* A, int lda,
         const float* B, int ldb, float beta, float* C, int ldc, const float* bias, cudaStream_t stream, int prof_kind) {
  ProfScope prof(prof_kind, 2.0 * M * N * K, stream);
  if (mode == GEMM_BF16) mode = GEMM_TF32;      // only the discriminator's big contractions have bf16 operands
  if (mode != GEMM_FP32) {
    bool handled = false;
    int rc = GIC_OK;
    if (mode == GEMM_TF32) {
      rc = gemm_tc_persistent(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, stream, &handled);
      if (rc != GIC_OK) return rc;
      if (handled) return GIC_OK;
    }
    rc = gemm_tc(mode, transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, stream, &handled);
    if (rc != GIC_OK) return rc;
    if (handled) return GIC_OK;
  }
  return gemm_f32(transA, transB, M, N, K, alpha, A, lda, B, ldb, beta, C, ldc, bias, stream);
}

}  // namespace gic
