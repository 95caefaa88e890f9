// GEMM machinery shared by the decoder relevance (decoder.cu) and the decoder gradient (decoder_grad.cu) kernels:
// an fp32 CUDA-core SGEMM with fused epilogues, the error-compensated bf16x3 tensor-core GEMM through lrpx_tc_conv, and
// the small helpers both files use.
#pragma once
#include "lrpx_common.cuh"

#include <algorithm>

namespace lrpx {

// ------------------------------------------------------------------------------------------------
// SGEMM  C[M,N] = A[M,K] @ B[K,N]  (row-major), 64x64x16 tiles, 4x4 per thread, fused epilogues.
// ------------------------------------------------------------------------------------------------
enum { GE_STORE = 0, GE_FEAT = 1, GE_AOA_PROJ = 2, GE_ADD = 3, GE_ADD_MASK = 4 };

struct GemmEpi {
  // GE_FEAT: out[m][n] = feat[b][p][n] * (acc + add_q[q][n])      rows m = q*P + p
  // GE_AOA_PROJ: out[m][n] = (A[b][p][n] * (acc + add_q[q][n])) / stab(A_pre[b][p][n])
  // GE_ADD: out[m][n] = add_q[q][n] + acc                         (gradient of the projector, gridTDmodel.py:1500-1502)
  // GE_ADD_MASK: as GE_ADD where feat[b][p][n] > 0, else 0         (guided variant, :1674)
  const float* x0;       // feat / A          (B,P,N)
  const float* x1;       // A_pre             (B,P,N)
  const float* add_q;    // (Q,N) or null
  const int32_t* req_img;
  int P;
};

template <int EPI>
__global__ void __launch_bounds__(256) sgemm_nn_kernel(const float* __restrict__ A, const float* __restrict__ Bm,
                                                       float* __restrict__ C, int M, int N, int K, int lda, int ldb,
                                                       int ldc, GemmEpi e) {
  constexpr int TBM = 64, TBN = 64, TBK = 16;
  __shared__ float As[TBK][TBM + 4];
  __shared__ float Bs[TBK][TBN];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  // 1-D grid, column tiles fastest: M / 64 row tiles exceed the 65 535 blocks of a grid's y dimension at Q * P rows
  const int ntn = (N + TBN - 1) / TBN;
  const int mt = blockIdx.x / ntn;
  const int m0 = mt * TBM, n0 = (blockIdx.x - mt * ntn) * TBN;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += TBK) {
#pragma unroll
    for (int j = 0; j < 4; ++j) {           // A tile: 64 x 16
      int idx = tid + 256 * j;
      int r = idx / TBK, c = idx % TBK;
      int m = m0 + r, k = k0 + c;
      As[c][r] = (m < M && k < K) ? A[(size_t)m * lda + k] : 0.f;
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {           // B tile: 16 x 64
      int idx = tid + 256 * j;
      int r = idx / TBN, c = idx % TBN;
      int k = k0 + r, n = n0 + c;
      Bs[r][c] = (k < K && n < N) ? Bm[(size_t)k * ldb + n] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < TBK; ++kk) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = Bs[kk][tx + 16 * j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + ty * 4 + i;
    if (m >= M) continue;
    int q = 0, pp = 0, b = 0;
    if (EPI != GE_STORE) {
      q = m / e.P;
      pp = m % e.P;
      b = e.req_img[q];
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tx + 16 * j;
      if (n >= N) continue;
      float v = acc[i][j];
      if (EPI == GE_FEAT) {
        float add = e.add_q ? e.add_q[(size_t)q * N + n] : 0.f;
        v = e.x0[((size_t)b * e.P + pp) * N + n] * (v + add);
      } else if (EPI == GE_ADD || EPI == GE_ADD_MASK) {
        float add = e.add_q ? e.add_q[(size_t)q * N + n] : 0.f;
        v = add + v;
        if (EPI == GE_ADD_MASK && !(e.x0[((size_t)b * e.P + pp) * N + n] > 0.f)) v = 0.f;
      } else if (EPI == GE_AOA_PROJ) {
        size_t o = ((size_t)b * e.P + pp) * N + n;
        float add = e.add_q ? e.add_q[(size_t)q * N + n] : 0.f;
        v = (e.x0[o] * (v + add)) / stab(e.x1[o]);
      }
      C[(size_t)m * ldc + n] = v;
    }
  }
}

template <int EPI>
static int sgemm(const float* A, const float* B, float* C, int M, int N, int K, const GemmEpi& e, cudaStream_t st) {
  if (M == 0) return LRPX_OK;
  const unsigned grid = (unsigned)ceil_div(N, 64) * (unsigned)ceil_div(M, 64);
  sgemm_nn_kernel<EPI><<<grid, 256, 0, st>>>(A, B, C, M, N, K, K, N, N, e);
  cudaError_t err = cudaGetLastError();
  if (err != cudaSuccess) {
    set_error("sgemm launch failed: %s", cudaGetErrorString(err));
    return LRPX_E_CUDA;
  }
  return LRPX_OK;
}

// ------------------------------------------------------------------------------------------------
// Error-compensated tensor-core GEMM (LRPX_DEC_TC_GEMM):  x = hi + lo with hi = bf16(x), lo = bf16(x - hi);
//   a*w ~= a_hi*w_hi + a_hi*w_lo + a_lo*w_hi   (the dropped lo*lo term is ~2^-16 relative)
// evaluated as ONE bf16 GEMM with the K dimension concatenated three times, fp32 accumulation in TMEM:
//   A' = [a_hi | a_hi | a_lo]  (M x 3K),   W' = [w_hi | w_lo | w_hi]  (N x 3K, K-major = the transposed weight)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void split_bf16(float x, __nv_bfloat16& hi, __nv_bfloat16& lo) {
  hi = __float2bfloat16(x);
  lo = __float2bfloat16(x - __bfloat162float(hi));
}
// bf16 elements of the split operand of a GEMM with `rows` rows and reduction length K: each row is stored [hi | lo]
// (2K), the layout put_operand, split3_act_kernel and the attention kernels' SPLIT stores write.  The GEMM reads it as
// [hi | lo | hi] (a_phys = 2K in gemm_any).  Every workspace slot that receives a split operand is sized by this rule.
static inline size_t split_elems(size_t rows, size_t K) { return rows * 2 * K; }
// a producer kernel writes its GEMM operand both as fp32 (CUDA-core GEMM) and, when `a3` is given, directly as the
// split row [hi | lo] of the tensor-core GEMM (saves the separate split pass over the operand)
__device__ __forceinline__ void put_operand(float* u, __nv_bfloat16* a3, size_t row, int K, int k, float x) {
  u[row * K + k] = x;
  if (a3) {
    __nv_bfloat16 hi, lo;
    split_bf16(x, hi, lo);
    __nv_bfloat16* o = a3 + row * 2 * K;
    o[k] = hi; o[K + k] = lo;
  }
}
// rows x K fp32 (row pitch lda) -> rows x 2K bf16 [hi | lo]; the GEMM reads a row as K = [hi | lo | hi] (a_phys wrap of
// lrpx_tc_conv: the third block group re-reads the first), so hi is stored once: 2/3 of the bytes of [hi | hi | lo]
static __global__ void split3_act_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ out, long long rows, int K,
                                  int lda) {
  long long total = rows * K;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long r = i / K;
    int k = (int)(i - r * K);
    __nv_bfloat16 hi, lo;
    split_bf16(x[r * lda + k], hi, lo);
    __nv_bfloat16* o = out + r * 2 * K;
    o[k] = hi; o[K + k] = lo;
  }
}
// W (K x N fp32 row-major, i.e. [k][n]) -> N x 3K bf16 [hi | hi | lo] of W^T:  a*w ~ a_hi*w_hi + a_lo*w_hi + a_hi*w_lo
static __global__ void split3_weight_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ out, int K, int N) {
  long long total = (long long)K * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int n = (int)(i % N);
    int k = (int)(i / N);
    __nv_bfloat16 hi, lo;
    split_bf16(w[i], hi, lo);
    __nv_bfloat16* o = out + (size_t)n * 3 * K;
    o[k] = hi; o[K + k] = hi; o[2 * K + k] = lo;
  }
}
// GE_FEAT / GE_AOA_PROJ epilogues applied to a plain GEMM result in place
template <int EPI>
__global__ void gemm_epilogue_kernel(float* __restrict__ C, long long M, int N, GemmEpi e) {
  long long total = M * N;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long m = i / N;
    int n = (int)(i - m * N);
    int q = (int)(m / e.P), pp = (int)(m % e.P);
    int b = e.req_img[q];
    size_t o = ((size_t)b * e.P + pp) * N + n;
    float add = e.add_q ? e.add_q[(size_t)q * N + n] : 0.f;
    float v;
    if (EPI == GE_ADD || EPI == GE_ADD_MASK) {
      v = add + C[i];
      if (EPI == GE_ADD_MASK && !(e.x0[o] > 0.f)) v = 0.f;
    } else {
      v = e.x0[o] * (C[i] + add);
      if (EPI == GE_AOA_PROJ) v = v / stab(e.x1[o]);
    }
    C[i] = v;
  }
}

static inline int ew_grid(long long total) {
  long long g = (total + 255) / 256, cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}
static bool tc_shape_ok(int N, int K) { return K % 64 == 0 && N % 32 == 0 && (N <= 256 || N % 256 == 0); }

// C[M,N] = A[M,K] @ W[K,N] (+ epilogue): tensor cores when `wt3` (prepared W') is given, CUDA cores otherwise
// a3_ready: the producer kernel already wrote the split operand [hi | lo] into a3 (no fp32 A exists then)
template <int EPI>
static int gemm_any(const float* A, const float* W, const __nv_bfloat16* wt3, __nv_bfloat16* a3, float* C, int M, int N,
                    int K, const GemmEpi& e, cudaStream_t st, bool a3_ready = false) {
  if (M == 0) return LRPX_OK;
  if (!wt3) return sgemm<EPI>(A, W, C, M, N, K, e, st);
  if (!a3_ready) split3_act_kernel<<<ew_grid((long long)M * K), 256, 0, st>>>(A, a3, M, K, K);
  lrpx_tc_conv_args g{};
  g.cin = 3 * K; g.a_phys = 2 * K; g.ncol = N; g.ksize = 1;
  g.a = a3; g.wt = wt3; g.out = C;
  if (EPI == GE_STORE) {          // one PF "block" of M rows: the STORE_F32 epilogue writes every in-range row
    g.n_img = 1; g.h = 0; g.w = M - 1;
    g.epilogue = LRPX_TC_EPI_STORE_F32;
    return lrpx_tc_conv(&g, st);
  }
  if (EPI == GE_ADD || EPI == GE_ADD_MASK) {      // plain store, then the addend / mask pass in place
    g.n_img = 1; g.h = 0; g.w = M - 1;
    g.epilogue = LRPX_TC_EPI_STORE_F32;
    int rc = lrpx_tc_conv(&g, st);
    if (rc != LRPX_OK) return rc;
    gemm_epilogue_kernel<EPI><<<ew_grid((long long)M * N), 256, 0, st>>>(C, M, N, e);
    return LRPX_OK;
  }
  // projector rules fused into the GEMM's epilogue: rows are (request, pixel) = one PF "block" of P rows per request
  g.n_img = M / e.P; g.h = 0; g.w = e.P - 1;
  g.epilogue = EPI == GE_FEAT ? LRPX_TC_EPI_FEAT : LRPX_TC_EPI_FEAT_DIV;
  g.x = e.x0; g.x1 = e.x1; g.bias = e.add_q; g.row_img = e.req_img;
  return lrpx_tc_conv(&g, st);
}
// Route of the GEMM with weight W (K x N): the prepared copy W' written into dst (N x 3K) when `tc` is set and the
// tensor cores take the shape, null when the GEMM stays on the CUDA cores.
// ready: dst still holds the split copy of W from an earlier call on the same workspace (LRPX_DEC_W3_READY)
static const __nv_bfloat16* tc_weight(bool tc, const float* W, __nv_bfloat16* dst, int K, int N, cudaStream_t st,
                                      bool ready = false) {
  if (!tc || !tc_shape_ok(N, K)) return nullptr;
  if (!ready) split3_weight_kernel<<<ew_grid((long long)K * N), 256, 0, st>>>(W, dst, K, N);
  return dst;
}

// r_words / max|r_words|   (:1129-1132)
static __global__ void words_norm_kernel(float* r_words, const int32_t* req_t, int T) {
  int q = blockIdx.x;
  int t = req_t[q];
  float* r = r_words + (size_t)q * T;
  float m = 0.f;
  for (int i = threadIdx.x; i <= t; i += 32) m = fmaxf(m, fabsf(r[i]));
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (m > 0.f)
    for (int i = threadIdx.x; i <= t; i += 32) r[i] = r[i] / m;
}

// block-wide sum of `v` written by thread 0 through `store`
template <class F>
__device__ __forceinline__ void block_sum_store(float v, F store) {
  for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  __shared__ float sm[32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  if (lane == 0) sm[wid] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    float s = 0.f;
    for (int k = 0; k < (blockDim.x + 31) / 32; ++k) s += sm[k];
    store(s);
  }
}
// Word relevance of request q, for the args struct of any decoder entry point: r_words (Q x T) and, when given,
// r_words_raw hold the same values until words_norm_kernel normalises r_words.  Words past t stay zero.
template <class Args>
__device__ __forceinline__ void zero_words(const Args& a, int q) {
  for (int j = threadIdx.x; j < a.T; j += blockDim.x) {
    a.r_words[(size_t)q * a.T + j] = 0.f;
    if (a.r_words_raw) a.r_words_raw[(size_t)q * a.T + j] = 0.f;
  }
}
template <class Args>
__device__ __forceinline__ void store_word(const Args& a, int q, int i, float s) {
  a.r_words[(size_t)q * a.T + i] = s;
  if (a.r_words_raw) a.r_words_raw[(size_t)q * a.T + i] = s;
}

static size_t align_up(size_t x) { return (x + 63) & ~(size_t)63; }
// Walks a workspace layout slot by slot, each slot starting on an align_up boundary: with a null base it only sizes the
// workspace (the *_workspace_bytes entry points), with the caller's base it places the slots.
struct Carver {
  float* base;
  size_t off = 0;          // floats
  float* f32(size_t n) {
    float* p = base ? base + off : nullptr;
    off += align_up(n);
    return p;
  }
  __nv_bfloat16* bf16(size_t n) { return reinterpret_cast<__nv_bfloat16*>(f32((n + 1) / 2)); }
  size_t bytes() const { return off * sizeof(float); }
};

}  // namespace lrpx
