// Fused element-wise steps of the explainer's teacher-forced forward (the producer of the saved state the decoder
// relevance kernels consume), fp32.
//
//   ExplainGridTDAttention.get_hidden_parameters   models/gridTDmodel.py:933-1012
//     adalstm_forward / language_lstm_forward      :773-797   (hand-rolled LSTM cells returning g, i, f)
//     AdaptiveAttention.forward                    :61-103    (adaptive attention with the sentinel)
//
// The reference runs ~30 small tensor ops per time step.  Here a step is: one GEMM over the concatenated
// recurrent inputs (library GEMM on the host side), lrpx_lstm_cell_f32, one GEMM for the two attention
// projections, lrpx_adaptive_attention_f32, one GEMM, lrpx_lstm_cell_f32.  Outputs go straight into the
// (B, T, .) saved-state tensors (row strides) and into the staging rows of the next GEMM.
#include "lrpx_common.cuh"

namespace lrpx {

__device__ __forceinline__ float sigmoidf_(float x) { return 1.f / (1.f + expf(-x)); }

// z: (B, >=4H) pre-activations in torch's gate order i, f, g, o (gridTDmodel.py:777-783)
__global__ void lstm_cell_kernel(lrpx_lstm_cell_args a) {
  const int b = blockIdx.y;
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= a.H) return;
  const float* z = a.z + (size_t)b * a.ldz;
  const float zi = z[j], zf = z[a.H + j], zg = z[2 * a.H + j], zo = z[3 * a.H + j];
  const float i = sigmoidf_(zi), f = sigmoidf_(zf);
  const float c = f * a.c_prev[(size_t)b * a.ld_cprev + j] + i * tanhf(zg);
  const float tc = tanhf(c);
  const float og = sigmoidf_(zo);
  const float h = og * tc;
  a.h[(size_t)b * a.ld_state + j] = h;
  a.c[(size_t)b * a.ld_state + j] = c;
  a.g[(size_t)b * a.ld_gate + j] = zg;
  a.i[(size_t)b * a.ld_gate + j] = i;
  a.f[(size_t)b * a.ld_gate + j] = f;
  if (a.o) a.o[(size_t)b * a.ld_gate + j] = og;
  if (a.h_copy0) a.h_copy0[(size_t)b * a.ld_copy0 + j] = h;
  if (a.h_copy1) a.h_copy1[(size_t)b * a.ld_copy1 + j] = h;
  if (a.h_copy2) a.h_copy2[(size_t)b * a.ld_copy2 + j] = h;
  if (a.gate_pre) {      // sentinel  s = sigmoid(x_gate(x) + h_gate(h_old)) * tanh(c_new)   (:982-983)
    const float sgv = sigmoidf_(a.gate_pre[(size_t)b * a.ld_gate_pre + j]);
    const float s = sgv * tc;
    a.s[(size_t)b * a.ld_gate + j] = s;
    if (a.sg) a.sg[(size_t)b * a.ld_gate + j] = sgv;
    if (a.s_copy) a.s_copy[(size_t)b * a.ld_s_copy + j] = s;
  }
}

// ------------------------------------------------------------------------------------------------
// LSTM step = skinny GEMM + cell update.  CTA = 4 hidden units x G gates (4*G weight rows of K floats, contiguous in
// the prepared layout) x a tile of 64 batch rows; the K-slices' partial sums meet in shared memory and slice 0 applies
// the cell rule.  fp32 throughout (the saved state feeds the fp32 decoder relevance).
// ------------------------------------------------------------------------------------------------
constexpr int LS_U = 4, LS_ROWS = 64, LS_SLICES = 8, LS_RPT = 8;
// K chunk / ring depth are template parameters of the step kernel (see lrpx_lstm_step_f32)

__global__ void lstm_prep_weights_kernel(const float* __restrict__ w, float* __restrict__ wp, int K, int G, int H) {
  const long long total = (long long)K * G * H;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    const long long r = i / K;                 // ((ug * G) + g) * 4 + u
    const int u = (int)(r % LS_U), g = (int)((r / LS_U) % G), ug = (int)(r / (LS_U * G));
    wp[i] = w[(size_t)k * G * H + (size_t)g * H + ug * LS_U + u];
  }
}

__device__ __forceinline__ void cp_async16(float* smem_dst, const float* gsrc, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
  const int n = valid ? 16 : 0;                 // src-size 0: the 16 bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(n) : "memory");
}

// 256 threads = 8 K-slices (one warp each) x (8 row groups x 4 units); a thread owns rows {rg + 8 i, i < 8} of one
// unit: per 4 k it reads 8 + G float4 from shared memory for 32*G FMAs.  K chunks of 64 go through a 4-stage cp.async
// ring: a CTA only moves ~0.35 MB, so what has to be covered is the L2 latency (measured: one chunk of look-ahead left
// the kernel at 22 us, no faster than the library GEMM it replaces).
template <int G, int LS_KC, int LS_STAGES>
__global__ void __launch_bounds__(256) lstm_step_kernel(lrpx_lstm_step_args a) {
  constexpr int LS_PITCH = LS_KC + 4;
  extern __shared__ __align__(16) float ls_smem[];
  constexpr int XS = LS_ROWS * LS_PITCH, WS = G * LS_U * LS_PITCH;
  float* xs = ls_smem;                               // [LS_STAGES][LS_ROWS][LS_PITCH]
  float* ws = xs + LS_STAGES * XS;                   // [LS_STAGES][G*4][LS_PITCH]
  float* red = ws + LS_STAGES * WS;                  // [8 slices][8 rows][G][32 lanes] partial sums
  const int tid = threadIdx.x, ks = tid >> 5, lane = tid & 31, rg = lane >> 2, u = lane & 3;
  const int ug = blockIdx.x, j = ug * LS_U + u, H = a.H, K = a.K;
  const float* wsrc = a.wp + (size_t)ug * G * LS_U * K;
  const int nchunk = (K + LS_KC - 1) / LS_KC;
  for (int row0 = 0; row0 < a.B; row0 += LS_ROWS) {
    auto issue = [&](int c) {
      const int k0 = c * LS_KC;
      float* xd = xs + (c % LS_STAGES) * XS;
      float* wd = ws + (c % LS_STAGES) * WS;
      for (int idx = tid; idx < LS_ROWS * (LS_KC / 4); idx += 256) {
        const int r = idx / (LS_KC / 4), c4 = (idx % (LS_KC / 4)) * 4;
        const bool ok = row0 + r < a.B && k0 + c4 < K;
        cp_async16(xd + r * LS_PITCH + c4, ok ? a.x + (size_t)(row0 + r) * a.ldx + k0 + c4 : a.x, ok);
      }
      for (int idx = tid; idx < G * LS_U * (LS_KC / 4); idx += 256) {
        const int r = idx / (LS_KC / 4), c4 = (idx % (LS_KC / 4)) * 4;
        const bool ok = k0 + c4 < K;
        cp_async16(wd + r * LS_PITCH + c4, ok ? wsrc + (size_t)r * K + k0 + c4 : wsrc, ok);
      }
    };
    // this thread's cell (row rg + 8*ks): its addend and previous cell state, fetched before the K loop
    float addv[G], cprev = 0.f;
    {
      const int bb = row0 + rg + 8 * ks;
#pragma unroll
      for (int g = 0; g < G; ++g) addv[g] = bb < a.B ? a.add[(size_t)bb * a.ld_add + (size_t)g * H + j] : 0.f;
      if (bb < a.B) cprev = a.c_prev[(size_t)bb * a.ld_cprev + j];
    }
    float acc[LS_RPT][G];
#pragma unroll
    for (int i = 0; i < LS_RPT; ++i)
#pragma unroll
      for (int g = 0; g < G; ++g) acc[i][g] = 0.f;
    __syncthreads();                                  // the previous row tile is done with the ring
    for (int c = 0; c < LS_STAGES - 1; ++c) {         // one commit group per chunk slot, empty past the end
      if (c < nchunk) issue(c);
      asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (int c = 0; c < nchunk; ++c) {
      if (c + LS_STAGES - 1 < nchunk) issue(c + LS_STAGES - 1);      // refills the stage computed in iteration c-1
      asm volatile("cp.async.commit_group;" ::: "memory");
      asm volatile("cp.async.wait_group %0;" ::"n"(LS_STAGES - 1) : "memory");
      __syncthreads();
      const float* xc = xs + (c % LS_STAGES) * XS;
      const float* wc = ws + (c % LS_STAGES) * WS;
      const int kb = ks * (LS_KC / LS_SLICES);
#pragma unroll
      for (int kk = kb; kk < kb + LS_KC / LS_SLICES; kk += 4) {
        float4 wv[G];
#pragma unroll
        for (int g = 0; g < G; ++g) wv[g] = *reinterpret_cast<const float4*>(wc + (g * LS_U + u) * LS_PITCH + kk);
#pragma unroll
        for (int i = 0; i < LS_RPT; ++i) {
          const float4 xv = *reinterpret_cast<const float4*>(xc + (rg + 8 * i) * LS_PITCH + kk);
#pragma unroll
          for (int g = 0; g < G; ++g) {
            acc[i][g] = fmaf(xv.x, wv[g].x, acc[i][g]);
            acc[i][g] = fmaf(xv.y, wv[g].y, acc[i][g]);
            acc[i][g] = fmaf(xv.z, wv[g].z, acc[i][g]);
            acc[i][g] = fmaf(xv.w, wv[g].w, acc[i][g]);
          }
        }
      }
      __syncthreads();                                // this stage is refilled by the next iteration's issue
    }
    // Sum the eight K-slices through shared memory ([slice][row i][gate][lane]: conflict-free both ways); thread
    // (ks, lane) then finishes ONE cell: row rg + 8*ks of its unit, so the transcendental-heavy cell rule runs on all
    // 256 threads (on slice 0 alone it was a quarter of the kernel's time).
#pragma unroll
    for (int i = 0; i < LS_RPT; ++i)
#pragma unroll
      for (int g = 0; g < G; ++g) red[((ks * LS_RPT + i) * G + g) * 32 + lane] = acc[i][g];
    __syncthreads();
    const int b = row0 + rg + 8 * ks;
    if (b < a.B) {
      float z[G];
#pragma unroll
      for (int g = 0; g < G; ++g) {
        float v = 0.f;
#pragma unroll
        for (int sl = 0; sl < LS_SLICES; ++sl) v += red[((sl * LS_RPT + ks) * G + g) * 32 + lane];
        z[g] = v + addv[g];
      }
      const float ig = sigmoidf_(z[0]), fg = sigmoidf_(z[1]);
      const float c = fg * cprev + ig * tanhf(z[2]);
      const float tc = tanhf(c);
      const float og = sigmoidf_(z[3]);
      const float h = og * tc;
      a.h[(size_t)b * a.ld_state + j] = h;
      a.c[(size_t)b * a.ld_state + j] = c;
      a.g[(size_t)b * a.ld_gate + j] = z[2];
      a.i[(size_t)b * a.ld_gate + j] = ig;
      a.f[(size_t)b * a.ld_gate + j] = fg;
      if (a.o) a.o[(size_t)b * a.ld_gate + j] = og;
      if (a.h_copy0) a.h_copy0[(size_t)b * a.ld_copy0 + j] = h;
      if (a.h_copy1) a.h_copy1[(size_t)b * a.ld_copy1 + j] = h;
      if (a.h_copy2) a.h_copy2[(size_t)b * a.ld_copy2 + j] = h;
      if (G == 5) {
        const float sgv = sigmoidf_(z[G - 1]);
        const float sv = sgv * tc;
        a.s[(size_t)b * a.ld_gate + j] = sv;
        if (a.sg) a.sg[(size_t)b * a.ld_gate + j] = sgv;
        if (a.s_copy) a.s_copy[(size_t)b * a.ld_s_copy + j] = sv;
      }
    }
  }
}

// One block per image.  AdaptiveAttention.attend (gridTDmodel.py:80-103):
//   z[p]   = sum_k w_h[k] * tanh(img_proj[b][p][k] + hproj[b][p])     (sic: the reference adds the h projection
//            along the pixel axis — its bmm with a ones matrix, :81-87 — which is only shape-valid for P == K, Q19)
//   alpha  = softmax_p z;  ctx = sum_p alpha[p] * A[b][p][:]
//   zs     = sum_k w_h[k] * tanh(sproj[b][k] + hproj[b][k]);  beta = softmax([z ; zs])[-1]
//   ctx_hat = beta * s + (1 - beta) * ctx
// The kernel moves 0.55 MB per image (img_proj 0.15 MB, A 0.4 MB, both L2-resident over the time steps) and is bound
// by how many of those bytes it keeps in flight: 1024 threads, three score rows (21 loads per lane) at a time in
// phase 1, float4 loads over four pixel groups (partial sums met in shared memory) in phase 3.
constexpr int AT_THREADS = 1024;
__global__ void __launch_bounds__(AT_THREADS) adaptive_attention_kernel(lrpx_ada_attention_args a) {
  extern __shared__ __align__(16) float sm[];            // z[P] | hproj[K] | sproj[K] | w_h[K] | red[32] | part[<=8][H]
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = blockDim.x >> 5;
  const int P = a.P, K = a.K, H = a.H;
  float* z = sm;
  float* hp = z + ((P + 3) & ~3);
  float* sp = hp + ((K + 3) & ~3);
  float* wh = sp + ((K + 3) & ~3);
  float* red = wh + ((K + 3) & ~3);
  float* part = red + 32;
  for (int k = tid; k < K; k += blockDim.x) wh[k] = a.w_h[k];
  if (a.hs_proj) {
    for (int k = tid; k < K; k += blockDim.x) {
      hp[k] = a.hs_proj[(size_t)b * a.ld_hs + k];
      sp[k] = a.hs_proj[(size_t)b * a.ld_hs + K + k];
    }
  } else {
    // hp = W_g_proj(h) (no bias), sp = W_s_proj(s) + b_s  (gridTDmodel.py:80,89): one warp per output, lanes over H
    const float* hv = a.h + (size_t)b * a.ld_h;
    const float* sv = a.s + (size_t)b * a.ld_s;
    for (int o = warp; o < 2 * K; o += nwarp) {
      const bool is_s = o >= K;
      const int k = is_s ? o - K : o;
      const float* wrow = (is_s ? a.W_s : a.W_g) + (size_t)k * H;
      const float* xv = is_s ? sv : hv;
      float acc = 0.f;
      for (int j = lane; j < H; j += 32) acc += wrow[j] * xv[j];
      for (int of = 16; of; of >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, of);
      if (lane == 0) {
        if (is_s) sp[k] = acc + a.b_s[k]; else hp[k] = acc;
      }
    }
  }
  __syncthreads();
  // ---- phase 1: scores.  Row P is the sentinel.  Rows p, p + nwarp, p + 2 nwarp of a warp are loaded together.
  const float* ip = a.img_proj + (size_t)b * P * K;
  constexpr int KI = 8;                                    // supports K <= 256 with every load issued up front
  if (K <= 32 * KI) {
    for (int p0 = warp; p0 <= P; p0 += 3 * nwarp) {
      float v[3][KI];
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int p = p0 + r * nwarp;
#pragma unroll
        for (int i = 0; i < KI; ++i) {
          const int k = lane + 32 * i;
          v[r][i] = (p < P && k < K) ? __ldg(ip + (size_t)p * K + k) : 0.f;
        }
      }
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const int p = p0 + r * nwarp;
        if (p > P) continue;
        const float hpp = p < P ? hp[p] : 0.f;     // Q19: the h projection is broadcast along the PIXEL axis here (:81-87)
        float acc = 0.f;
#pragma unroll
        for (int i = 0; i < KI; ++i) {
          const int k = lane + 32 * i;
          if (k < K) acc += wh[k] * tanhf(p < P ? v[r][i] + hpp : sp[k] + hp[k]);
        }
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
          if (p < P) z[p] = acc; else red[31] = acc;
        }
      }
    }
  } else {
    for (int p = warp; p <= P; p += nwarp) {
      float acc = 0.f;
      if (p < P) {
        const float hpp = hp[p];
        for (int k = lane; k < K; k += 32) acc += wh[k] * tanhf(__ldg(ip + (size_t)p * K + k) + hpp);
      } else {
        for (int k = lane; k < K; k += 32) acc += wh[k] * tanhf(sp[k] + hp[k]);
      }
      for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
      if (lane == 0) {
        if (p < P) z[p] = acc; else red[31] = acc;
      }
    }
  }
  __syncthreads();
  const float zs = red[31];
  __syncthreads();
  // ---- phase 2: softmax over the P pixel scores; the sentinel joins for the second softmax
  float m = -INFINITY;
  for (int p = tid; p < P; p += blockDim.x) m = fmaxf(m, z[p]);
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if (lane == 0) red[warp] = m;
  __syncthreads();
  m = -INFINITY;
  for (int w = 0; w < nwarp; ++w) m = fmaxf(m, red[w]);
  __syncthreads();
  float sum = 0.f;
  for (int p = tid; p < P; p += blockDim.x) sum += expf(z[p] - m);
  for (int o = 16; o; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = 0.f;
  for (int w = 0; w < nwarp; ++w) sum += red[w];
  __syncthreads();
  const float m2 = fmaxf(m, zs);
  const float sum2 = sum * expf(m - m2) + expf(zs - m2);
  const float beta = expf(zs - m2) / sum2;
  for (int p = tid; p < P; p += blockDim.x) {
    const float al = expf(z[p] - m) / sum;
    z[p] = al;
    a.alpha[(size_t)b * a.ld_alpha + p] = al;
  }
  if (tid == 0) a.beta[(size_t)b * a.ld_beta] = beta;
  __syncthreads();
  // ---- phase 3: ctx[h] = sum_p alpha[p] A[p][h]; thread = (pixel group pg, four consecutive h), float4 loads
  const float* A = a.A + (size_t)b * P * H;
  const int hq = H >> 2;                                   // float4 columns
  if ((H & 3) == 0 && 4 * hq <= (int)blockDim.x) {
    const int pg = tid / hq, h4 = tid - pg * hq;
    const int ngroups = min(8, (int)blockDim.x / hq);     // pixel groups whose partial sums meet in `part`
    if (pg < ngroups) {
      float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
      const int per = (P + ngroups - 1) / ngroups, pb = pg * per, pe = min(P, pb + per);
      int p = pb;
      for (; p + 7 <= pe; p += 7) {
        float4 av[7];
#pragma unroll
        for (int q = 0; q < 7; ++q) av[q] = __ldg(reinterpret_cast<const float4*>(A + (size_t)(p + q) * H) + h4);
#pragma unroll
        for (int q = 0; q < 7; ++q) {
          const float al = z[p + q];
          acc.x += av[q].x * al; acc.y += av[q].y * al; acc.z += av[q].z * al; acc.w += av[q].w * al;
        }
      }
      for (; p < pe; ++p) {
        const float4 av = __ldg(reinterpret_cast<const float4*>(A + (size_t)p * H) + h4);
        const float al = z[p];
        acc.x += av.x * al; acc.y += av.y * al; acc.z += av.z * al; acc.w += av.w * al;
      }
      *reinterpret_cast<float4*>(part + (size_t)pg * H + 4 * h4) = acc;
    }
    __syncthreads();
    for (int h = tid; h < H; h += blockDim.x) {
      float acc = 0.f;
      for (int g = 0; g < ngroups; ++g) acc += part[(size_t)g * H + h];
      const float s = a.s[(size_t)b * a.ld_s + h];
      const float ch = beta * s + (1.f - beta) * acc;
      a.ctx[(size_t)b * a.ld_out + h] = acc;
      a.ctx_hat[(size_t)b * a.ld_out + h] = ch;
      if (a.ctx_hat_copy) a.ctx_hat_copy[(size_t)b * a.ld_copy + h] = ch;
    }
  } else {
    for (int h = tid; h < H; h += blockDim.x) {
      float acc = 0.f;
      for (int p = 0; p < P; ++p) acc += __ldg(A + (size_t)p * H + h) * z[p];
      const float s = a.s[(size_t)b * a.ld_s + h];
      const float ch = beta * s + (1.f - beta) * acc;
      a.ctx[(size_t)b * a.ld_out + h] = acc;
      a.ctx_hat[(size_t)b * a.ld_out + h] = ch;
      if (a.ctx_hat_copy) a.ctx_hat_copy[(size_t)b * a.ld_copy + h] = ch;
    }
  }
}

}  // namespace lrpx

using namespace lrpx;

extern "C" int lrpx_lstm_cell_f32(const lrpx_lstm_cell_args* a, void* stream) {
  LRPX_CHECK_ARG(a && a->B > 0 && a->H > 0, "bad shape");
  LRPX_CHECK_ARG(a->z && a->c_prev && a->h && a->c && a->g && a->i && a->f, "null pointer");
  LRPX_CHECK_ARG(!a->gate_pre || a->s, "gate_pre needs the sentinel output s");
  dim3 grid(ceil_div(a->H, 128), a->B);
  lstm_cell_kernel<<<grid, 128, 0, as_stream(stream)>>>(*a);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

extern "C" int lrpx_lstm_prep_weights_f32(const float* w, float* wp, int K, int G, int H, void* stream) {
  LRPX_CHECK_ARG(w && wp && K > 0 && (G == 4 || G == 5) && H > 0 && H % LS_U == 0, "bad argument (G in {4,5}, H % 4 == 0)");
  const long long total = (long long)K * G * H;
  long long grid = (total + 255) / 256;
  if (grid > 148 * 16) grid = 148 * 16;
  lstm_prep_weights_kernel<<<(int)grid, 256, 0, as_stream(stream)>>>(w, wp, K, G, H);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

extern "C" int lrpx_lstm_step_f32(const lrpx_lstm_step_args* a, void* stream) {
  LRPX_CHECK_ARG(a && a->B > 0 && a->H > 0 && a->H % LS_U == 0 && a->K > 0 && a->K % 4 == 0 && (a->G == 4 || a->G == 5),
                 "bad shape (H % 4 == 0, K % 4 == 0, G in {4,5})");
  LRPX_CHECK_ARG(a->x && a->wp && a->add && a->c_prev && a->h && a->c && a->g && a->i && a->f, "null pointer");
  LRPX_CHECK_ARG(a->G == 4 || a->s, "G == 5 needs the sentinel output s");
  LRPX_CHECK_ARG(a->ldx % 4 == 0 && (reinterpret_cast<uintptr_t>(a->x) & 15) == 0 &&
                     (reinterpret_cast<uintptr_t>(a->wp) & 15) == 0,
                 "x rows and wp must be 16-byte aligned");
  cudaStream_t st = as_stream(stream);
  // K chunk x ring depth: 256 x 2 by default — measured for the explainer's two shapes (K = 1024 / 5 gates, K = 1536 /
  // 4 gates, 64 rows): 64 x 4: 19.0 / 23.4 us, 128 x 3: 17.0 / 21.3 us, 256 x 2: 15.5 / 20.5 us (fewer block-wide
  // barriers, one 87 KB chunk of look-ahead).  LRPX_LSTM_KC = 64 | 128 select the other variants.
  static const int kc = [] { const char* e = getenv("LRPX_LSTM_KC"); const int v = e ? atoi(e) : 256;
                             return (v == 64 || v == 128) ? v : 256; }();
  auto launch = [&](auto kernel, int KC, int STAGES, std::atomic<uint64_t>& done) {
    const size_t smem = (size_t)(STAGES * (LS_ROWS * (KC + 4) + a->G * LS_U * (KC + 4)) + LS_SLICES * 32 * LS_RPT * a->G) * sizeof(float);
    const int rc = ensure_smem_attr(kernel, (int)smem, done);
    if (rc == LRPX_OK) kernel<<<a->H / LS_U, 256, smem, st>>>(*a);
    return rc;
  };
  static std::atomic<uint64_t> attr_done[6];
  int rc;
  if (kc == 128) {
    if (a->G == 5) rc = launch(lstm_step_kernel<5, 128, 3>, 128, 3, attr_done[0]);
    else rc = launch(lstm_step_kernel<4, 128, 3>, 128, 3, attr_done[1]);
  } else if (kc == 256) {
    if (a->G == 5) rc = launch(lstm_step_kernel<5, 256, 2>, 256, 2, attr_done[4]);
    else rc = launch(lstm_step_kernel<4, 256, 2>, 256, 2, attr_done[5]);
  } else {
    if (a->G == 5) rc = launch(lstm_step_kernel<5, 64, 4>, 64, 4, attr_done[2]);
    else rc = launch(lstm_step_kernel<4, 64, 4>, 64, 4, attr_done[3]);
  }
  if (rc != LRPX_OK) return rc;
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

extern "C" int lrpx_adaptive_attention_f32(const lrpx_ada_attention_args* a, void* stream) {
  LRPX_CHECK_ARG(a && a->B > 0 && a->P > 0 && a->K > 0 && a->H > 0, "bad shape");
  LRPX_CHECK_ARG(a->P == a->K, "the reference's attention is only defined for P == n_pixel (gridTDmodel.py:81-87)");
  LRPX_CHECK_ARG(a->A && a->img_proj && a->w_h && a->s && a->ctx && a->ctx_hat && a->alpha && a->beta, "null pointer");
  LRPX_CHECK_ARG(a->hs_proj || (a->h && a->W_g && a->W_s && a->b_s), "hs_proj or (h, W_g, W_s, b_s) required");
  const int hq = a->H / 4;
  const int groups = (a->H % 4 == 0 && 4 * hq <= AT_THREADS) ? (AT_THREADS / hq < 8 ? AT_THREADS / hq : 8) : 0;
  size_t smem = (size_t)(((a->P + 3) & ~3) + 3 * ((a->K + 3) & ~3) + 32 + groups * a->H) * sizeof(float);
  LRPX_CHECK_ARG(smem <= 48 * 1024, "P + 3K + H too large for one block");
  adaptive_attention_kernel<<<a->B, AT_THREADS, smem, as_stream(stream)>>>(*a);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}
