// Decoder part of the gradient-family explainers (SURVEY.md §8 f4), batched over Q = (image, target word) requests.
//
//   gridTD : ExplainGridTDGradient.explain_caption_wordt          models/gridTDmodel.py:1424-1508
//            ExplainiGridTDGuidedGradient.explain_caption_wordt   models/gridTDmodel.py:1588-1675
//   AoA    : ExplainAOAGradient.explain_caption_wordt             models/aoamodel.py:1435-1499 (+ gradient_mha :1415-1433)
//   CAM    : grad_cam                                             models/gridTDmodel.py:1760-1771, aoamodel.py:1676-1689
//
// The reference hand-writes the backward pass of its decoder with the attention weights, the sentinel gate and the
// attention-on-attention gate held constant, one vector at a time.  Like the relevance kernels of decoder.cu, a step i
// (t..0) here is: an element-wise kernel forming the four gate derivatives of all requests, ONE (Q x 4H) @ (4H x in)
// GEMM, an element-wise kernel distributing the slices of its result.  Reference quirks kept:
//   * d_h1t[i+1] is OVERWRITTEN by the language LSTM's input slice (:1482), so the AdaLSTM's own recurrent term
//     d_gates1 @ W_hh (:1494) never reaches anything: that GEMM is not computed;
//   * AoA: d_global_img_feature is ASSIGNED per step (aoamodel.py:1488), the value of step 0 survives;
//   * the guided variant's masks on ReLU outputs compare with `< 0` (:1663,:1665) and never fire; the mask on the
//     encoder output (`<= 0`, :1674) does.
#include "lrpx_common.cuh"
#include "dec_gemm.cuh"

namespace lrpx {

// LSTM cell backward for one unit (gridTDmodel.py:1463-1472): dh = gradient of h_{i+1}, dc = gradient already carried
// by c_{i+1}.  Returns the four gate pre-activation gradients (order i, f, g, o) and the carry into c_i.
struct CellGrad { float di, df, dg, dov, dc_prev; };
__device__ __forceinline__ CellGrad cell_backward(float dh, float dc_in, float c_new, float c_old, float g_pre, float ig,
                                                  float fg, float og) {
  const float tc = tanhf(c_new);
  const float d_o_act = dh * tc;
  const float dc = dc_in + dh * og * (1.f - tc * tc);
  const float ga = tanhf(g_pre);
  const float d_f_act = dc * c_old;
  const float d_i_act = dc * ga;
  const float d_g_act = dc * ig;
  CellGrad r;
  r.dc_prev = dc * fg;
  r.di = d_i_act * ig * (1.f - ig);
  r.df = d_f_act * fg * (1.f - fg);
  r.dov = d_o_act * og * (1.f - og);
  r.dg = d_g_act * (1.f - ga * ga);
  return r;
}
__device__ __forceinline__ void put_gates(float* u, __nv_bfloat16* a3, size_t q, int H, int j, const CellGrad& g) {
  put_operand(u, a3, q, 4 * H, j, g.di);
  put_operand(u, a3, q, 4 * H, H + j, g.df);
  put_operand(u, a3, q, 4 * H, 2 * H + j, g.dg);
  put_operand(u, a3, q, 4 * H, 3 * H + j, g.dov);
}
__device__ __forceinline__ void zero_gates(float* u, __nv_bfloat16* a3, size_t q, int H, int j) {
  for (int k = 0; k < 4; ++k) put_operand(u, a3, q, 4 * H, k * H + j, 0.f);
}

// ------------------------------------------------------------------------------------------------
// gridTD
// ------------------------------------------------------------------------------------------------
struct GGradWs {
  float *d_h2, *d_c2, *d_c1, *d_glob, *u, *v, *uctx, *coefavg, *dproj;
  __nv_bfloat16 *a3, *a3u, *w3_2, *w3_1, *w3_glob, *w3_proj;
};

__global__ void ggrad_init_kernel(lrpx_gridtd_grad_args a, GGradWs w) {
  const int q = blockIdx.x;
  const float* wr = a.W_fc + (size_t)a.req_word[q] * a.H;      // d logits[word] / d (ctx_hat + h2) = W_fc[word]  (:1459)
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    const size_t o = (size_t)q * a.H + j;
    w.d_h2[o] = wr[j];
    w.d_c2[o] = 0.f;
    w.d_c1[o] = 0.f;
  }
  for (int j = threadIdx.x; j < a.E; j += blockDim.x) w.d_glob[(size_t)q * a.E + j] = 0.f;
  zero_words(a, q);
}
// LanguageLSTM cell backward (:1463-1473) -> u = [d_i | d_f | d_g | d_o]
__global__ void ggrad_cell2_kernel(lrpx_gridtd_grad_args a, GGradWs w, int i) {
  const int q = blockIdx.x, H = a.H;
  const int b = a.req_img[q], t = a.req_t[q];
  const size_t bi = ((size_t)b * a.T + i) * H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * H, bi0 = bi1 - H;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    if (i > t) { zero_gates(w.u, w.a3u, q, H, j); continue; }
    const size_t o = (size_t)q * H + j;
    const CellGrad g = cell_backward(w.d_h2[o], w.d_c2[o], a.c2[bi1 + j], a.c2[bi0 + j], a.g2[bi + j], a.i2[bi + j],
                                     a.f2[bi + j], a.o2[bi + j]);
    w.d_c2[o] = g.dc_prev;
    put_gates(w.u, w.a3u, q, H, j, g);
  }
}
// after v = u @ [W_ih2 | W_hh2]: slices [ctx_hat | h1 | h2] (:1474-1482), sentinel / context split, AdaLSTM cell backward
__global__ void ggrad_post2_kernel(lrpx_gridtd_grad_args a, GGradWs w, int i) {
  const int q = blockIdx.x, H = a.H;
  const int b = a.req_img[q], t = a.req_t[q];
  const size_t bi = ((size_t)b * a.T + i) * H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * H, bi0 = bi1 - H;
  const float* vq = w.v + (size_t)q * 3 * H;
  const float* wr = a.W_fc + (size_t)a.req_word[q] * H;
  const float beta = i <= t ? a.beta[(size_t)b * a.T + i] : 0.f;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    if (i > t) { zero_gates(w.u, w.a3u, q, H, j); continue; }
    const size_t o = (size_t)q * H + j;
    const float d_cth = (i == t ? wr[j] : 0.f) + vq[j];                       // :1460, :1476
    w.uctx[((size_t)q * a.T + i) * H + j] = d_cth * (1.f - beta);              // d_context (:1477)
    const float d_st = d_cth * beta;                                           // :1480
    const float c1n = a.c1[bi1 + j];
    const float tc = tanhf(c1n);
    const float dc_in = w.d_c1[o] + d_st * a.sg[bi + j] * (1.f - tc * tc);     // :1481
    const CellGrad g = cell_backward(vq[H + j], dc_in, c1n, a.c1[bi0 + j], a.g1[bi + j], a.i1[bi + j], a.f1[bi + j],
                                     a.o1[bi + j]);                            // d_h1t[i+1] = d_x2t[i][H:]  (:1482)
    w.d_c1[o] = g.dc_prev;
    put_gates(w.u, w.a3u, q, H, j, g);
    w.d_h2[o] = vq[2 * H + j];                                                 // :1474
  }
}
// after v = u @ W_ih1: slices [h2 | glob | emb] (:1495-1498)
__global__ void ggrad_post1_kernel(lrpx_gridtd_grad_args a, GGradWs w, int i) {
  const int q = blockIdx.x, H = a.H, E = a.E;
  if (i > a.req_t[q]) return;
  const float* vq = w.v + (size_t)q * (H + 2 * E);
  float wsum = 0.f;
  for (int k = threadIdx.x; k < H + 2 * E; k += blockDim.x) {
    const float d = vq[k];
    if (k < H) w.d_h2[(size_t)q * H + k] += d;
    else if (k < H + E) w.d_glob[(size_t)q * E + (k - H)] += d;
    else wsum += d;
  }
  block_sum_store(wsum, [&](float s) { store_word(a, q, i, s); });            // :1503
}
// coefavg = (d_glob @ W_glob) / P    (:1499, :1501)
__global__ void ggrad_avg_kernel(lrpx_gridtd_grad_args a, GGradWs w) {
  const int q = blockIdx.x;
  for (int c = threadIdx.x; c < a.C; c += blockDim.x)
    w.coefavg[(size_t)q * a.C + c] = 1.0f * w.v[(size_t)q * a.C + c] / (float)a.P;
}
// d_img_feature_proj[q][p][h] = sum_{i = t..0} alpha_i[p] * d_context_i[h]   (:1478-1479): one block per request, the
// request's alpha rows and d_context rows in shared memory, four hidden units per thread (H % 4 == 0), pixels four at
// a time.  SPLIT: the result leaves as the [hi | lo] operand of the tensor-core projector GEMM.
template <bool SPLIT>
__global__ void __launch_bounds__(512) ggrad_attn_kernel(const float* __restrict__ alpha, const float* __restrict__ uctx,
                                                         const int32_t* __restrict__ req_img,
                                                         const int32_t* __restrict__ req_t, float* __restrict__ dproj,
                                                         __nv_bfloat16* __restrict__ a3, int T, int P, int H) {
  extern __shared__ __align__(16) float gatt_s[];          // alpha[(t+1)][P4] | uctx[(t+1)][H]
  const int q = blockIdx.x;
  const int b = req_img[q], t = req_t[q];
  const int P4 = (P + 3) & ~3;
  float* al_s = gatt_s;
  float* u_s = gatt_s + (size_t)(t + 1) * P4;
  for (int k = threadIdx.x; k < (t + 1) * P4; k += blockDim.x) {
    const int i = k / P4, p = k - i * P4;
    al_s[k] = p < P ? alpha[((size_t)b * T + i) * P + p] : 0.f;
  }
  for (int k = threadIdx.x; k < (t + 1) * H; k += blockDim.x) u_s[k] = uctx[(size_t)q * T * H + k];
  __syncthreads();
  for (int h4 = threadIdx.x * 4; h4 < H; h4 += blockDim.x * 4) {
    for (int p0 = 0; p0 < P; p0 += 4) {
      float acc[4][4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[k][j] = 0.f;
      for (int i = t; i >= 0; --i) {
        const float4 uv = *reinterpret_cast<const float4*>(u_s + i * H + h4);
        const float4 a4 = *reinterpret_cast<const float4*>(al_s + i * P4 + p0);
        const float al[4] = {a4.x, a4.y, a4.z, a4.w}, uu[4] = {uv.x, uv.y, uv.z, uv.w};
#pragma unroll
        for (int k = 0; k < 4; ++k)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[k][j] = fmaf(uu[j], al[k], acc[k][j]);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (p0 + k >= P) break;
        const size_t row = (size_t)q * P + p0 + k;
        if (SPLIT) {
          uint32_t hi2[2], lo2[2];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            __nv_bfloat16 h0, l0, h1, l1;
            split_bf16(acc[k][2 * j], h0, l0);
            split_bf16(acc[k][2 * j + 1], h1, l1);
            hi2[j] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
            lo2[j] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
          }
          __nv_bfloat16* o = a3 + row * 2 * H + h4;
          *reinterpret_cast<uint2*>(o) = make_uint2(hi2[0], hi2[1]);
          *reinterpret_cast<uint2*>(o + H) = make_uint2(lo2[0], lo2[1]);
        } else {
          *reinterpret_cast<float4*>(dproj + row * H + h4) = make_float4(acc[k][0], acc[k][1], acc[k][2], acc[k][3]);
        }
      }
    }
  }
}

// the same sum, one block per (pixel, request): for captions too long for the shared-memory form above
template <bool SPLIT>
__global__ void ggrad_attn_slow_kernel(const float* __restrict__ alpha, const float* __restrict__ uctx,
                                       const int32_t* __restrict__ req_img, const int32_t* __restrict__ req_t,
                                       float* __restrict__ dproj, __nv_bfloat16* __restrict__ a3, int T, int P, int H) {
  const int q = blockIdx.x / P, p = blockIdx.x - q * P;            // one block per (request, pixel)
  const int b = req_img[q], t = req_t[q];
  const float* al = alpha + (size_t)b * T * P + p;
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    float acc = 0.f;
    for (int i = t; i >= 0; --i) acc = fmaf(uctx[((size_t)q * T + i) * H + h], al[(size_t)i * P], acc);
    if (SPLIT) put_operand(dproj, a3, (size_t)q * P + p, H, h, acc);
    else dproj[((size_t)q * P + p) * H + h] = acc;
  }
}

static size_t ggrad_carve(const lrpx_gridtd_grad_args* a, float* base, GGradWs* w) {
  Carver c{base};
  const size_t Q = a->Q, H = a->H, E = a->E, C = a->C;
  size_t nmax = 3 * H > H + 2 * E ? 3 * H : H + 2 * E;
  if (C > nmax) nmax = C;
  GGradWs t{};
  t.d_h2 = c.f32(Q * H); t.d_c2 = c.f32(Q * H); t.d_c1 = c.f32(Q * H);
  t.d_glob = c.f32(Q * E);
  t.u = c.f32(Q * 4 * H);
  t.v = c.f32(Q * nmax);
  t.uctx = c.f32(Q * a->T * H);
  t.coefavg = c.f32(Q * C);
  t.dproj = c.f32(Q * a->P * H);
  if (a->flags & LRPX_DEC_TC_GEMM) {
    // a3: W_proj (Q*P, H), W_glob (Q, E), W2 and W1 (Q, 4H) unless fused;  a3u: W2 and W1 fused (Q, 4H)
    t.a3 = c.bf16(std::max({split_elems(Q * a->P, H), split_elems(Q, E), split_elems(Q, 4 * H)}));
    t.a3u = c.bf16(split_elems(Q, 4 * H));
    t.w3_2 = c.bf16(3 * H * 3 * 4 * H);
    t.w3_1 = c.bf16((H + 2 * E) * 3 * 4 * H);
    t.w3_glob = c.bf16(C * 3 * E);
    t.w3_proj = c.bf16(C * 3 * H);
  }
  if (w) *w = t;
  return c.bytes();
}

// ------------------------------------------------------------------------------------------------
// AoA
// ------------------------------------------------------------------------------------------------
struct AGradWs {
  float *d_h, *d_c, *d_glob, *uA, *uB, *u, *v, *dval, *dproj;
  __nv_bfloat16 *a3, *w3_aoa, *w3_gate, *w3_g, *w3_v, *w3_proj;
};

__device__ __forceinline__ float sigmoid_(float x) { return 1.f / (1.f + expf(-x)); }

// fc, then the attention-on-attention product  ctx_aoa = sigmoid(gate) * linear   (aoamodel.py:1462-1468)
__global__ void agrad_init_kernel(lrpx_aoa_grad_args a, AGradWs w) {
  const int q = blockIdx.x, H = a.H;
  const int b = a.req_img[q], t = a.req_t[q];
  const float* wr = a.W_fc + (size_t)a.req_word[q] * H;
  const size_t bt = ((size_t)b * a.T + t) * H;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    const size_t o = (size_t)q * H + j;
    const float d0 = wr[j];
    const float sg = sigmoid_(a.caoa_gate[bt + j]);
    w.d_h[o] = d0;
    w.d_c[o] = 0.f;
    w.uA[o] = d0 * sg;
    w.uB[o] = d0 * a.caoa_lin[bt + j] * (1.f - sg) * sg;
  }
  zero_words(a, q);
}
// d_h[t+1] += d_B @ W_gate  (:1470);  d_value[p] = d_context (.) alpha[head][p] on the chosen head (gradient_mha :1415-1433)
__global__ void agrad_ctx_kernel(lrpx_aoa_grad_args a, AGradWs w, const float* __restrict__ v_ctx,
                                 const float* __restrict__ v_gate, __nv_bfloat16* a3) {
  const int q = blockIdx.x / a.P, p = blockIdx.x - q * a.P, H = a.H;     // one block per (request, pixel)
  const int b = a.req_img[q], t = a.req_t[q], head = a.req_head[q];
  const int dk = H / a.num_head;
  const float al = a.alpha[(((size_t)b * a.T + t) * a.num_head + head) * a.P + p];
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    const float dv = (h / dk == head) ? v_ctx[(size_t)q * H + h] * al : 0.f;
    put_operand(w.dval, a3, (size_t)q * a.P + p, H, h, dv);
    if (p == 0) w.d_h[(size_t)q * H + h] += v_gate[(size_t)q * H + h];
  }
}
__global__ void agrad_cell_kernel(lrpx_aoa_grad_args a, AGradWs w, int i) {
  const int q = blockIdx.x, H = a.H;
  const int b = a.req_img[q], t = a.req_t[q];
  const size_t bi = ((size_t)b * a.T + i) * H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * H, bi0 = bi1 - H;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    if (i > t) { zero_gates(w.u, nullptr, q, H, j); continue; }
    const size_t o = (size_t)q * H + j;
    const CellGrad g = cell_backward(w.d_h[o], w.d_c[o], a.c[bi1 + j], a.c[bi0 + j], a.g[bi + j], a.i[bi + j],
                                     a.f[bi + j], a.o[bi + j]);
    w.d_c[o] = g.dc_prev;
    put_gates(w.u, nullptr, q, H, j, g);
  }
}
// after v = u @ [W_ih | W_hh]: slices [emb | glob | h] (:1486-1489)
__global__ void agrad_post_kernel(lrpx_aoa_grad_args a, AGradWs w, int i) {
  const int q = blockIdx.x, H = a.H, E = a.E;
  if (i > a.req_t[q]) return;
  const float* vq = w.v + (size_t)q * (E + 2 * H);
  float wsum = 0.f;
  for (int k = threadIdx.x; k < E + 2 * H; k += blockDim.x) {
    const float d = vq[k];
    if (k < E) wsum += d;
    else if (k < E + H) { if (i == 0) w.d_glob[(size_t)q * H + (k - E)] = d / (float)a.P; }   // assigned, step 0 survives
    else w.d_h[(size_t)q * H + (k - E - H)] = d;
  }
  block_sum_store(wsum, [&](float s) { store_word(a, q, i, s); });
}

static size_t agrad_carve(const lrpx_aoa_grad_args* a, float* base, AGradWs* w) {
  Carver c{base};
  const size_t Q = a->Q, H = a->H, E = a->E;
  AGradWs t{};
  t.d_h = c.f32(Q * H); t.d_c = c.f32(Q * H); t.d_glob = c.f32(Q * H);
  t.uA = c.f32(Q * H); t.uB = c.f32(Q * H);
  t.u = c.f32(Q * 4 * H);
  t.v = c.f32(Q * (E + 2 * H));
  t.dval = c.f32(Q * a->P * H);
  t.dproj = c.f32(Q * a->P * H);
  if (a->flags & LRPX_DEC_TC_GEMM) {
    // a3: W_v and W_proj (Q*P, H), W_g (Q, 4H), W_aoa and W_gate (Q, H)
    t.a3 = c.bf16(std::max({split_elems(Q * a->P, H), split_elems(Q, 4 * H), split_elems(Q, H)}));
    t.w3_aoa = c.bf16(H * 3 * H);
    t.w3_gate = c.bf16(H * 3 * H);
    t.w3_g = c.bf16((E + 2 * H) * 3 * 4 * H);
    t.w3_v = c.bf16(H * 3 * H);
    t.w3_proj = c.bf16((size_t)a->C * 3 * H);
  }
  if (w) *w = t;
  return c.bytes();
}

// ------------------------------------------------------------------------------------------------
// Adaptive attention (single AdaLSTM): ExplainAdaptiveGradient.explain_caption_wordt, adaptiveattention.py:965-1021.
// The reference applies the attention / sentinel split ONLY at the explained step t (:987-994, outside its loop); the
// loop then walks the LSTM alone.  d_img_feature_proj = d_context (x) alpha_t is rank one, so the projector needs one
// (Q x H) @ (H x C) GEMM and an outer-product kernel instead of a GEMM over all Q * P rows.
// ------------------------------------------------------------------------------------------------
struct DGradWs {
  float *d_h, *d_c, *d_glob, *dctx, *u, *v, *y;
  __nv_bfloat16 *a3, *w3_g, *w3_glob, *w3_proj;
};

__global__ void dgrad_init_kernel(lrpx_adaptive_grad_args a, DGradWs w) {
  const int q = blockIdx.x, H = a.H;
  const int b = a.req_img[q], t = a.req_t[q];
  const float* wr = a.W_fc + (size_t)a.req_word[q] * H;
  const float beta = a.beta[(size_t)b * a.T + t];
  const size_t bt = ((size_t)b * a.T + t) * H, bt1 = ((size_t)b * (a.T + 1) + t + 1) * H;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    const size_t o = (size_t)q * H + j;
    const float d0 = wr[j];                                                    // :987
    const float tc = tanhf(a.c[bt1 + j]);
    w.dctx[o] = d0 * (1.f - beta);                                             // :989
    w.d_c[o] = d0 * beta * a.sg[bt + j] * (1.f - tc * tc);                     // :990-991
    w.d_h[o] = d0;                                                             // :992
  }
  for (int j = threadIdx.x; j < a.E; j += blockDim.x) w.d_glob[(size_t)q * a.E + j] = 0.f;
  zero_words(a, q);
}
__global__ void dgrad_cell_kernel(lrpx_adaptive_grad_args a, DGradWs w, int i) {
  const int q = blockIdx.x, H = a.H;
  const int b = a.req_img[q], t = a.req_t[q];
  const size_t bi = ((size_t)b * a.T + i) * H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * H, bi0 = bi1 - H;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    if (i > t) { zero_gates(w.u, nullptr, q, H, j); continue; }
    const size_t o = (size_t)q * H + j;
    const CellGrad g = cell_backward(w.d_h[o], w.d_c[o], a.c[bi1 + j], a.c[bi0 + j], a.g[bi + j], a.i[bi + j],
                                     a.f[bi + j], a.o[bi + j]);
    w.d_c[o] = g.dc_prev;
    put_gates(w.u, nullptr, q, H, j, g);
  }
}
// after v = u @ [W_ih | W_hh]: slices [emb | glob | h] (:1007-1010)
__global__ void dgrad_post_kernel(lrpx_adaptive_grad_args a, DGradWs w, int i) {
  const int q = blockIdx.x, H = a.H, E = a.E;
  if (i > a.req_t[q]) return;
  const float* vq = w.v + (size_t)q * (2 * E + H);
  float wsum = 0.f;
  for (int k = threadIdx.x; k < 2 * E + H; k += blockDim.x) {
    const float d = vq[k];
    if (k < E) wsum += d;
    else if (k < 2 * E) w.d_glob[(size_t)q * E + (k - E)] += d;
    else w.d_h[(size_t)q * H + (k - 2 * E)] = d;
  }
  block_sum_store(wsum, [&](float s) { store_word(a, q, i, s); });
}
// d_feat[q][p][c] = (d_glob @ W_glob)[c] / P + alpha_t[p] * (d_context @ W_proj)[c]     (:1011-1015)
__global__ void dgrad_out_kernel(lrpx_adaptive_grad_args a, const float* __restrict__ avg /* (Q,C) */,
                                 const float* __restrict__ y /* (Q,C) */) {
  const int q = blockIdx.x / a.P, p = blockIdx.x - q * a.P;          // one block per (request, pixel)
  const int b = a.req_img[q], t = a.req_t[q];
  const float al = a.alpha[((size_t)b * a.T + t) * a.P + p];
  float* dst = a.d_feat + ((size_t)q * a.P + p) * a.C;
  for (int c = threadIdx.x; c < a.C; c += blockDim.x)
    dst[c] = 1.0f * avg[(size_t)q * a.C + c] / (float)a.P + al * y[(size_t)q * a.C + c];
}

static size_t dgrad_carve(const lrpx_adaptive_grad_args* a, float* base, DGradWs* w) {
  Carver c{base};
  const size_t Q = a->Q, H = a->H, E = a->E, C = a->C;
  size_t nmax = 2 * E + H > C ? 2 * E + H : C;
  DGradWs t{};
  t.d_h = c.f32(Q * H); t.d_c = c.f32(Q * H); t.d_glob = c.f32(Q * E); t.dctx = c.f32(Q * H);
  t.u = c.f32(Q * 4 * H);
  t.v = c.f32(Q * nmax);
  t.y = c.f32(Q * C);
  if (a->flags & LRPX_DEC_TC_GEMM) {
    // a3: W_g (Q, 4H), W_glob (Q, E), W_proj (Q, H)
    t.a3 = c.bf16(std::max({split_elems(Q, 4 * H), split_elems(Q, E), split_elems(Q, H)}));
    t.w3_g = c.bf16((2 * E + H) * 3 * 4 * H);
    t.w3_glob = c.bf16(C * 3 * E);
    t.w3_proj = c.bf16(C * 3 * H);
  }
  if (w) *w = t;
  return c.bytes();
}

// ------------------------------------------------------------------------------------------------
// Grad-CAM (gridTDmodel.py:1760-1771): weights[c] = mean_p grads[q][p][c];  cam[p] = relu(sum_c feat[b][p][c] weights[c]);
// out[q][p] = cam[p] / (max|cam| + 1e-6).  One block per request.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) grad_cam_kernel(const float* __restrict__ feat, const float* __restrict__ grads,
                                                       const int32_t* __restrict__ req_img, float* __restrict__ out, int P,
                                                       int C) {
  extern __shared__ float cam_s[];          // weights[C] | cam[P]
  float* wgt = cam_s;
  float* cam = cam_s + C;
  __shared__ float red[32];
  const int q = blockIdx.x;
  const int b = req_img ? req_img[q] : q;
  const float* g = grads + (size_t)q * P * C;
  const float* f = feat + (size_t)b * P * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float s = 0.f;
    for (int p = 0; p < P; ++p) s += g[(size_t)p * C + c];
    wgt[c] = s / (float)P;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
  float mx = 0.f;
  for (int p = wid; p < P; p += nw) {
    float s = 0.f;
    for (int c = lane; c < C; c += 32) s = fmaf(f[(size_t)p * C + c], wgt[c], s);
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    s = fmaxf(s, 0.f);
    if (lane == 0) cam[p] = s;
    mx = fmaxf(mx, s);
  }
  if (lane == 0) red[wid] = mx;
  __syncthreads();
  mx = 0.f;
  for (int k = 0; k < nw; ++k) mx = fmaxf(mx, red[k]);
  const float den = mx + 1e-6f;
  for (int p = threadIdx.x; p < P; p += blockDim.x) out[(size_t)q * P + p] = cam[p] / den;
}

// Guided Grad-CAM's last step (gridTDmodel.py:1826-1828): out[q][c][y][x] = g[q][c][y][x] * (K_h cam_q K_w^T)[y][x] with
// K the (H x h) / (W x w) matrices of skimage's pyramid_expand along one axis (bilinear resize + Gaussian, both
// separable: models/_gradient.py::expand_operator).  One block per (request, output row).
__global__ void __launch_bounds__(256) cam_expand_mul_kernel(const float* __restrict__ g, const float* __restrict__ cam,
                                                             const float* __restrict__ Kh, const float* __restrict__ Kw,
                                                             float* __restrict__ out, int C, int h, int w, int H, int W) {
  extern __shared__ float cam_row_s[];       // t[w] = sum_i Kh[y][i] * cam[i][:]
  const int q = blockIdx.y, y = blockIdx.x;
  for (int j = threadIdx.x; j < w; j += blockDim.x) {
    float s = 0.f;
    for (int i = 0; i < h; ++i) s = fmaf(Kh[(size_t)y * h + i], cam[((size_t)q * h + i) * w + j], s);
    cam_row_s[j] = s;
  }
  __syncthreads();
  for (int x = threadIdx.x; x < W; x += blockDim.x) {
    float v = 0.f;
    for (int j = 0; j < w; ++j) v = fmaf(Kw[(size_t)x * w + j], cam_row_s[j], v);
    for (int c = 0; c < C; ++c) {
      const size_t o = (((size_t)q * C + c) * H + y) * W + x;
      out[o] = g[o] * v;
    }
  }
}

}  // namespace lrpx

using namespace lrpx;

extern "C" {

size_t lrpx_gridtd_decoder_grad_workspace_bytes(const lrpx_gridtd_grad_args* a) {
  if (!a) return 0;
  return ggrad_carve(a, nullptr, nullptr);
}

int lrpx_gridtd_decoder_grad_f32(const lrpx_gridtd_grad_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->B > 0 && a->T > 0 && a->H > 0 && a->H % 4 == 0 && a->E > 0 && a->P > 0 && a->C > 0 && a->V > 0 &&
                     a->Q >= 0,
                 "bad dimensions (H must be a multiple of 4)");
  if (a->Q == 0) return LRPX_OK;
  LRPX_CHECK_ARG(a->c1 && a->c2 && a->g1 && a->i1 && a->f1 && a->o1 && a->g2 && a->i2 && a->f2 && a->o2 && a->sg &&
                     a->alpha && a->beta && a->W1 && a->W2 && a->W_fc && a->W_glob && a->W_proj && a->req_img &&
                     a->req_t && a->req_word && a->d_feat && a->r_words,
                 "null pointer in args");
  const bool guided = (a->flags & LRPX_DEC_GUIDED) != 0;
  LRPX_CHECK_ARG(!guided || a->feat, "the guided variant masks with the encoder output: feat required");
  GGradWs w;
  const size_t need = ggrad_carve(a, (float*)workspace, &w);
  LRPX_CHECK_ARG(workspace && workspace_bytes >= need, "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Q = a->Q, H = a->H, E = a->E, T = a->T, P = a->P, C = a->C;
  const int nt = H >= 256 ? 256 : 128;
  GemmEpi none{};
  const bool tc = (a->flags & LRPX_DEC_TC_GEMM) != 0;
  const __nv_bfloat16* w3_2 = tc_weight(tc, a->W2, w.w3_2, 4 * H, 3 * H, st);
  const __nv_bfloat16* w3_1 = tc_weight(tc, a->W1, w.w3_1, 4 * H, H + 2 * E, st);
  const __nv_bfloat16* w3_glob = tc_weight(tc, a->W_glob, w.w3_glob, E, C, st);
  const __nv_bfloat16* w3_proj = tc_weight(tc, a->W_proj, w.w3_proj, H, C, st);
  const bool fused_split = w3_2 && w3_1;      // the step kernels write the split operand themselves
  if (!fused_split) w.a3u = nullptr;
  __nv_bfloat16* a3_step = fused_split ? w.a3u : w.a3;
  ggrad_init_kernel<<<Q, nt, 0, st>>>(*a, w);
  cudaMemsetAsync(w.uctx, 0, (size_t)Q * T * H * sizeof(float), st);
  for (int i = T - 1; i >= 0; --i) {
    ggrad_cell2_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W2, w3_2, a3_step, w.v, Q, 3 * H, 4 * H, none, st, fused_split));
    ggrad_post2_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W1, w3_1, a3_step, w.v, Q, H + 2 * E, 4 * H, none, st, fused_split));
    ggrad_post1_kernel<<<Q, 256, 0, st>>>(*a, w, i);
  }
  RUN(gemm_any<GE_STORE>(w.d_glob, a->W_glob, w3_glob, w.a3, w.v, Q, C, E, none, st));
  ggrad_avg_kernel<<<Q, 128, 0, st>>>(*a, w);
  const size_t att_smem = (size_t)T * (((P + 3) & ~3) + H) * sizeof(float);
  if (att_smem <= 200 * 1024) {
    static std::atomic<uint64_t> attr_done[2];
    const int at = H / 4 >= 512 ? 512 : ((H / 4 + 31) & ~31);
    if (w3_proj) {
      RUN(ensure_smem_attr(ggrad_attn_kernel<true>, 200 * 1024, attr_done[1]));
      ggrad_attn_kernel<true><<<Q, at, att_smem, st>>>(a->alpha, w.uctx, a->req_img, a->req_t, w.dproj, w.a3, T, P, H);
    } else {
      RUN(ensure_smem_attr(ggrad_attn_kernel<false>, 200 * 1024, attr_done[0]));
      ggrad_attn_kernel<false><<<Q, at, att_smem, st>>>(a->alpha, w.uctx, a->req_img, a->req_t, w.dproj, w.a3, T, P, H);
    }
  } else {          // long captions x wide hidden state: alpha and d_context rows do not fit one block's shared memory
    const unsigned qp = (unsigned)Q * P;
    if (w3_proj) ggrad_attn_slow_kernel<true><<<qp, nt, 0, st>>>(a->alpha, w.uctx, a->req_img, a->req_t, w.dproj, w.a3, T, P, H);
    else ggrad_attn_slow_kernel<false><<<qp, nt, 0, st>>>(a->alpha, w.uctx, a->req_img, a->req_t, w.dproj, w.a3, T, P, H);
  }
  GemmEpi fe{a->feat, nullptr, w.coefavg, a->req_img, P};
  if (guided) RUN(gemm_any<GE_ADD_MASK>(w.dproj, a->W_proj, w3_proj, w.a3, a->d_feat, Q * P, C, H, fe, st, w3_proj != nullptr));
  else RUN(gemm_any<GE_ADD>(w.dproj, a->W_proj, w3_proj, w.a3, a->d_feat, Q * P, C, H, fe, st, w3_proj != nullptr));
  words_norm_kernel<<<Q, 32, 0, st>>>(a->r_words, a->req_t, T);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

size_t lrpx_aoa_decoder_grad_workspace_bytes(const lrpx_aoa_grad_args* a) {
  if (!a) return 0;
  return agrad_carve(a, nullptr, nullptr);
}

int lrpx_aoa_decoder_grad_f32(const lrpx_aoa_grad_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->B > 0 && a->T > 0 && a->H > 0 && a->E > 0 && a->P > 0 && a->C > 0 && a->V > 0 && a->Q >= 0 &&
                     a->num_head > 0 && a->H % a->num_head == 0,
                 "bad dimensions");
  if (a->Q == 0) return LRPX_OK;
  LRPX_CHECK_ARG(a->c && a->g && a->i && a->f && a->o && a->caoa_gate && a->caoa_lin && a->alpha && a->W_g && a->W_fc &&
                     a->W_aoa && a->W_gate && a->W_v && a->W_proj && a->req_img && a->req_t && a->req_word &&
                     a->req_head && a->d_feat && a->r_words,
                 "null pointer in args");
  AGradWs w;
  const size_t need = agrad_carve(a, (float*)workspace, &w);
  LRPX_CHECK_ARG(workspace && workspace_bytes >= need, "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Q = a->Q, H = a->H, E = a->E, T = a->T, P = a->P, C = a->C;
  const int nt = H >= 256 ? 256 : 128;
  GemmEpi none{};
  const bool tc = (a->flags & LRPX_DEC_TC_GEMM) != 0;
  const __nv_bfloat16* w3_aoa = tc_weight(tc, a->W_aoa, w.w3_aoa, H, H, st);
  const __nv_bfloat16* w3_gate = tc_weight(tc, a->W_gate, w.w3_gate, H, H, st);
  const __nv_bfloat16* w3_g = tc_weight(tc, a->W_g, w.w3_g, 4 * H, E + 2 * H, st);
  const __nv_bfloat16* w3_v = tc_weight(tc, a->W_v, w.w3_v, H, H, st);
  const __nv_bfloat16* w3_proj = tc_weight(tc, a->W_proj, w.w3_proj, H, C, st);
  agrad_init_kernel<<<Q, nt, 0, st>>>(*a, w);
  float* v_ctx = w.v;                       // (Q,H)
  float* v_gate = w.v + (size_t)Q * H;      // (Q,H)   (v holds Q*(E+2H) floats)
  RUN(gemm_any<GE_STORE>(w.uA, a->W_aoa, w3_aoa, w.a3, v_ctx, Q, H, H, none, st));
  RUN(gemm_any<GE_STORE>(w.uB, a->W_gate, w3_gate, w.a3, v_gate, Q, H, H, none, st));
  agrad_ctx_kernel<<<(unsigned)Q * P, nt, 0, st>>>(*a, w, v_ctx, v_gate, w3_v ? w.a3 : nullptr);
  // the value projection's input gradient is formed first: its split operand occupies a3 until that GEMM has run
  GemmEpi ge{nullptr, nullptr, w.d_glob, a->req_img, P};
  // d_glob is known only after the LSTM chain: run the chain on the CUDA-core/tensor-core step GEMMs with their own
  // operand buffer (u is split by gemm_any into a3 only after the value GEMM below has consumed it)
  RUN(gemm_any<GE_STORE>(w.dval, a->W_v, w3_v, w.a3, w.dproj, Q * P, H, H, none, st, w3_v != nullptr));
  for (int i = T - 1; i >= 0; --i) {
    agrad_cell_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W_g, w3_g, w.a3, w.v, Q, E + 2 * H, 4 * H, none, st));
    agrad_post_kernel<<<Q, 256, 0, st>>>(*a, w, i);
  }
  // d_img_feature_proj = d_value @ W_v + d_glob / P   (:1490-1492), then the projector (:1493)
  gemm_epilogue_kernel<GE_ADD><<<ew_grid((long long)Q * P * H), 256, 0, st>>>(w.dproj, (long long)Q * P, H, ge);
  RUN(gemm_any<GE_STORE>(w.dproj, a->W_proj, w3_proj, w.a3, a->d_feat, Q * P, C, H, none, st));
  words_norm_kernel<<<Q, 32, 0, st>>>(a->r_words, a->req_t, T);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

size_t lrpx_adaptive_decoder_grad_workspace_bytes(const lrpx_adaptive_grad_args* a) {
  if (!a) return 0;
  return dgrad_carve(a, nullptr, nullptr);
}

int lrpx_adaptive_decoder_grad_f32(const lrpx_adaptive_grad_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->B > 0 && a->T > 0 && a->H > 0 && a->E > 0 && a->P > 0 && a->C > 0 && a->V > 0 && a->Q >= 0,
                 "bad dimensions");
  if (a->Q == 0) return LRPX_OK;
  LRPX_CHECK_ARG(a->c && a->g && a->i && a->f && a->o && a->sg && a->alpha && a->beta && a->W_g && a->W_fc && a->W_glob &&
                     a->W_proj && a->req_img && a->req_t && a->req_word && a->d_feat && a->r_words,
                 "null pointer in args");
  DGradWs w;
  const size_t need = dgrad_carve(a, (float*)workspace, &w);
  LRPX_CHECK_ARG(workspace && workspace_bytes >= need, "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Q = a->Q, H = a->H, E = a->E, T = a->T, C = a->C;
  const int nt = H >= 256 ? 256 : 128;
  GemmEpi none{};
  const bool tc = (a->flags & LRPX_DEC_TC_GEMM) != 0;
  const __nv_bfloat16* w3_g = tc_weight(tc, a->W_g, w.w3_g, 4 * H, 2 * E + H, st);
  const __nv_bfloat16* w3_glob = tc_weight(tc, a->W_glob, w.w3_glob, E, C, st);
  const __nv_bfloat16* w3_proj = tc_weight(tc, a->W_proj, w.w3_proj, H, C, st);
  dgrad_init_kernel<<<Q, nt, 0, st>>>(*a, w);
  for (int i = T - 1; i >= 0; --i) {
    dgrad_cell_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W_g, w3_g, w.a3, w.v, Q, 2 * E + H, 4 * H, none, st));
    dgrad_post_kernel<<<Q, 256, 0, st>>>(*a, w, i);
  }
  RUN(gemm_any<GE_STORE>(w.d_glob, a->W_glob, w3_glob, w.a3, w.v, Q, C, E, none, st));      // d_average_img_feature
  RUN(gemm_any<GE_STORE>(w.dctx, a->W_proj, w3_proj, w.a3, w.y, Q, C, H, none, st));        // d_context @ W_proj
  dgrad_out_kernel<<<(unsigned)Q * a->P, 256, 0, st>>>(*a, w.v, w.y);
  words_norm_kernel<<<Q, 32, 0, st>>>(a->r_words, a->req_t, T);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_grad_cam_f32(const float* feat, const float* grads, const int32_t* req_img, float* out, int Q, int P, int C,
                      void* stream) {
  LRPX_CHECK_ARG(feat && grads && out && Q >= 0 && P > 0 && C > 0, "bad argument");
  LRPX_CHECK_ARG((size_t)(P + C) * sizeof(float) <= 48 * 1024, "P + C too large for one block");
  if (Q == 0) return LRPX_OK;
  grad_cam_kernel<<<Q, 256, (size_t)(P + C) * sizeof(float), as_stream(stream)>>>(feat, grads, req_img, out, P, C);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_cam_expand_mul_f32(const float* g, const float* cam, const float* Kh, const float* Kw, float* out, int Q, int C,
                            int h, int w, int H, int W, void* stream) {
  LRPX_CHECK_ARG(g && cam && Kh && Kw && out && Q >= 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "bad argument");
  LRPX_CHECK_ARG((size_t)w * sizeof(float) <= 48 * 1024 && H <= 65535 && Q <= 65535, "map too large");
  if (Q == 0) return LRPX_OK;
  cam_expand_mul_kernel<<<dim3(H, Q), 256, (size_t)w * sizeof(float), as_stream(stream)>>>(g, cam, Kh, Kw, out, C, h, w, H, W);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

}  // extern "C"
