// Decoder relevance (fp32), batched over Q = (image, target word) requests.
//
//   gridTD : ExplainGridTDAttention.explain_caption_wordt   models/gridTDmodel.py:1014-1135
//   AoA    : ExplainAOAAttention.explain_caption_wordt      models/aoamodel.py:1064-1156 (+ lrp_mha :812-862)
//   tune   : get_lrp_weight_step                            models/gridTDmodel.py:549-578, aoamodel.py:597-626
//
// The reference walks each vector with lrp_linear_eps (gridTDmodel.py:744-765), materialising
// `weight * input` (out x in) and `eye(H)` on every call.  Here the same arithmetic is in closed form:
//   ident(r,x,z) = x * r / stab(z)                     (weight = eye)
//   lin(r,x,z,W) = x * ((r / stab(z)) @ W)              (GEMM over all requests at once)
// The LSTM chain is sequential in the step index i (t..0) but independent across requests, so every
// step is: one warp-friendly element-wise kernel + one (Q x H) @ (H x in) GEMM + one element-wise kernel.
#include "lrpx_common.cuh"
#include "dec_gemm.cuh"

namespace lrpx {

// fc rule for the target word only (one-hot relevance): gridTDmodel.py:1033-1059
//   r_sum = s_in * W_fc[word] * logit/stab(logit);  r_a = a * r_sum / stab(s_in), r_b likewise
__device__ __forceinline__ void fc_split(float a, float b, float wrow, float coef, float& ra, float& rb) {
  float s_in = a + b;
  float r_sum = s_in * wrow * coef;
  float d = stab(s_in);
  ra = a * r_sum / d;
  rb = b * r_sum / d;
}

// ------------------------------------------------------------------------------------------------
// gridTD
// ------------------------------------------------------------------------------------------------
struct GridWs {
  float *r_h2, *r_c2, *r_c1, *r_cth, *r_glob, *u, *v, *uctx, *coefavg, *wproj;
  float* gA;               // A / stab(A_pre) per image (B x P x H), the attention rule's per-image factor
  // LRPX_DEC_TC_GEMM: split activations (largest GEMM) and prepared weights, bf16
  __nv_bfloat16 *a3, *w3_g2, *w3_g1, *w3_glob, *w3_proj;
  __nv_bfloat16* a3u;      // split form of u written by the step kernels themselves (null: CUDA-core GEMMs)
};

__global__ void grid_init_kernel(lrpx_gridtd_args a, GridWs w) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q], word = a.req_word[q];
  float logit = a.pred[((size_t)b * a.T + t) * a.V + word];
  float coef = logit / stab(logit);
  const float* h2 = a.h2 + ((size_t)b * (a.T + 1) + t + 1) * a.H;
  const float* ch = a.ctx_hat + ((size_t)b * a.T + t) * a.H;
  const float* wr = a.W_fc + (size_t)word * a.H;
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    float rh, rc;
    fc_split(h2[j], ch[j], wr[j], coef, rh, rc);
    size_t o = (size_t)q * a.H + j;
    w.r_h2[o] = rh;
    w.r_cth[o] = rc;
    w.r_c2[o] = 0.f;
    w.r_c1[o] = 0.f;
  }
  for (int j = threadIdx.x; j < a.E; j += blockDim.x) w.r_glob[(size_t)q * a.E + j] = 0.f;
  zero_words(a, q);
}

// LanguageLSTM cell rule (:1061-1069) -> u = r_g2 / stab(g2)
__global__ void grid_cell2_kernel(lrpx_gridtd_args a, GridWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  bool active = i <= t;
  size_t bi = ((size_t)b * a.T + i) * a.H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * a.H,
         bi0 = ((size_t)b * (a.T + 1) + i) * a.H;
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    size_t o = (size_t)q * a.H + j;
    if (!active) { put_operand(w.u, w.a3u, q, a.H, j, 0.f); continue; }
    float rc2 = w.r_c2[o] + w.r_h2[o];
    float d = stab(a.c2[bi1 + j]);
    float g = a.g2[bi + j];
    float r_g = a.i2[bi + j] * tanhf(g) * rc2 / d;
    w.r_c2[o] = a.f2[bi + j] * a.c2[bi0 + j] * rc2 / d;
    put_operand(w.u, w.a3u, q, a.H, j, r_g / stab(g));
  }
}

// after v = u @ W_g2 : slices of xh2 (:1070-1084), attention split, AdaLSTM cell rule (:1096-1105)
__global__ void grid_post2_kernel(lrpx_gridtd_args a, GridWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  bool active = i <= t;
  const int H = a.H;
  size_t bi = ((size_t)b * a.T + i) * H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * H,
         bi0 = ((size_t)b * (a.T + 1) + i) * H;
  const float* x2 = a.x2 + ((size_t)b * a.T + i) * 2 * H;
  const float* vq = w.v + (size_t)q * 3 * H;
  float beta = a.beta[(size_t)b * a.T + i];
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    size_t o = (size_t)q * H + j;
    if (!active) { put_operand(w.u, w.a3u, q, H, j, 0.f); continue; }
    float rx_ctx = x2[j] * vq[j];                 // xh2[:H]   = ctx_hat_i
    float rx_h1 = x2[H + j] * vq[H + j];          // xh2[H:2H] = h1_{i+1}
    float rx_h2 = a.h2[bi0 + j] * vq[2 * H + j];  // xh2[2H:]  = h2_i
    float rcth = (i == t ? w.r_cth[o] : 0.f) + rx_ctx;
    float cth = a.ctx_hat[bi + j];
    float dct = stab(cth);
    float r_s = beta * a.st[bi + j] * rcth / dct;
    float cx = a.ctx[bi + j];
    float r_ctx = cx * (1.f - beta) * rcth / dct;
    w.uctx[((size_t)q * a.T + i) * H + j] = r_ctx / stab(cx);
    float rc1 = w.r_c1[o] + r_s + rx_h1;
    float d = stab(a.c1[bi1 + j]);
    float g = a.g1[bi + j];
    float r_g = a.i1[bi + j] * tanhf(g) * rc1 / d;
    w.r_c1[o] = a.f1[bi + j] * a.c1[bi0 + j] * rc1 / d;
    put_operand(w.u, w.a3u, q, H, j, r_g / stab(g));
    w.r_h2[o] = rx_h2;
  }
}

// after v = u @ W_g1 : slices of xh1 (:1106-1115)
__global__ void grid_post1_kernel(lrpx_gridtd_args a, GridWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  if (i > t) return;
  const int H = a.H, E = a.E;
  const float* x1 = a.x1 + ((size_t)b * a.T + i) * (H + 2 * E);
  const float* vq = w.v + (size_t)q * (2 * H + 2 * E);
  float wsum = 0.f;
  for (int k = threadIdx.x; k < H + 2 * E; k += blockDim.x) {
    float rx = x1[k] * vq[k];
    if (k < H) w.r_h2[(size_t)q * H + k] += rx;
    else if (k < H + E) w.r_glob[(size_t)q * E + (k - H)] += rx;
    else wsum += rx;
  }
  // r_h1[i] = rx1[H+2E:] is dead: it is overwritten at step i-1 before being read (:1075 vs :1110)
  block_sum_store(wsum, [&](float s) { store_word(a, q, i, s); });
}

// u_g = r_glob / stab(glob_pre)   (:1116-1119)
__global__ void grid_glob_kernel(lrpx_gridtd_args a, GridWs w) {
  int q = blockIdx.x, b = a.req_img[q];
  for (int j = threadIdx.x; j < a.E; j += blockDim.x)
    w.u[(size_t)q * a.E + j] = w.r_glob[(size_t)q * a.E + j] / stab(a.glob_pre[(size_t)b * a.E + j]);
}
// coefavg = avg * v / stab(avg) / P  (mean-pool rule, :1121-1124; r_avg = avg * v)
__global__ void grid_avg_kernel(lrpx_gridtd_args a, GridWs w) {
  int q = blockIdx.x, b = a.req_img[q];
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    float av = a.avg[(size_t)b * a.C + c];
    float r_avg = av * w.v[(size_t)q * a.C + c];
    w.coefavg[(size_t)q * a.C + c] = r_avg / stab(av) / (float)a.P;
  }
}
// wproj[q][p][h] = A * (sum_i alpha_i[p] * uctx_i[h]) / stab(A_pre)     (:1091-1095 then :1125-1128)
__global__ void grid_attn_kernel(lrpx_gridtd_args a, GridWs w) {
  const int q = blockIdx.x / a.P, p = blockIdx.x - q * a.P;          // one block per (request, pixel)
  int b = a.req_img[q], t = a.req_t[q];
  const float* al = a.alpha + (size_t)b * a.T * a.P + p;
  size_t o0 = ((size_t)b * a.P + p) * a.H;
  for (int h = threadIdx.x; h < a.H; h += blockDim.x) {
    float acc = 0.f;
    for (int i = t; i >= 0; --i) acc += al[(size_t)i * a.P] * w.uctx[((size_t)q * a.T + i) * a.H + h] * a.A[o0 + h];
    w.wproj[((size_t)q * a.P + p) * a.H + h] = acc / stab(a.A_pre[o0 + h]);
  }
}
// Same rule, one block per request and one thread per hidden unit.  The request's alpha rows ((t+1) x P) and uctx
// rows ((t+1) x H) sit in shared memory; a thread walks the pixels four at a time: per step i one LDS (uctx) + one
// LDS.128 (four alphas, broadcast) feed four FMAs, i = t..0 like the reference loop, then
// wproj = A * acc / stab(A_pre).  (The per-(request, pixel) form above re-reads uctx 196 times and spends ~4
// instructions per multiply-add: 1.4 ms per 1216 requests; this form is bound by its 0.7 GB of output.)
// SPLIT: the result leaves directly as the split bf16 operand [hi | lo] of the tensor-core projector GEMM.
// G = A / stab(A_pre), once per image (B x P x H; every request of the image multiplies by it)
__global__ void grid_attn_gain_kernel(const float* __restrict__ A, const float* __restrict__ A_pre, float* __restrict__ G,
                                      size_t n4) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 x = __ldg(reinterpret_cast<const float4*>(A) + i), z = __ldg(reinterpret_cast<const float4*>(A_pre) + i);
    reinterpret_cast<float4*>(G)[i] = make_float4(x.x / stab(z.x), x.y / stab(z.y), x.z / stab(z.z), x.w / stab(z.w));
  }
}
template <bool SPLIT>
__global__ void __launch_bounds__(512, 2) grid_attn_rows_kernel(lrpx_gridtd_args a, GridWs w) {
  extern __shared__ __align__(16) float att_s[];          // alpha[(t+1)][P4] | uctx[(t+1)][H]
  const int q = blockIdx.x;
  const int b = a.req_img[q], t = a.req_t[q];
  const int H = a.H, P = a.P, P4 = (P + 3) & ~3;
  float* al_s = att_s;
  float* u_s = att_s + (size_t)(t + 1) * P4;
  if ((H & 3) == 0 && (P & 3) == 0 && ((reinterpret_cast<uintptr_t>(a.alpha) | reinterpret_cast<uintptr_t>(w.uctx)) & 15) == 0) {
    // 16-byte copies, four in flight per thread: the element-wise form was (t+1)(P+H)/blockDim dependent load -> store
    // rounds per thread (27 at t = 18), each a trip to L2 — a third of the block's time before its first multiply
    const int p4 = P >> 2, n_al = (t + 1) * p4, n_u = (t + 1) * (H >> 2);
    float4* al4 = reinterpret_cast<float4*>(al_s);
    float4* u4 = reinterpret_cast<float4*>(u_s);
    const float4* usrc = reinterpret_cast<const float4*>(w.uctx + (size_t)q * a.T * H);
#pragma unroll 4
    for (int k = threadIdx.x; k < n_al; k += blockDim.x) {
      const int i = k / p4, c = k - i * p4;
      al4[k] = __ldg(reinterpret_cast<const float4*>(a.alpha + ((size_t)b * a.T + i) * P) + c);
    }
#pragma unroll 4
    for (int k = threadIdx.x; k < n_u; k += blockDim.x) u4[k] = usrc[k];
  } else {
    for (int k = threadIdx.x; k < (t + 1) * P4; k += blockDim.x) {
      const int i = k / P4, p = k - i * P4;
      al_s[k] = p < P ? a.alpha[((size_t)b * a.T + i) * P + p] : 0.f;
    }
    for (int k = threadIdx.x; k < (t + 1) * H; k += blockDim.x) u_s[k] = w.uctx[(size_t)q * a.T * H + k];
  }
  __syncthreads();
  if ((H & 3) == 0) {
    // four hidden units x four pixels per thread step: per LSTM step one LDS.128 of uctx and one of the alphas feed 16
    // FMAs; the per-image factor G = A / stab(A_pre) (grid_attn_gain_kernel) comes in 16-byte loads issued before the
    // loop, the results leave as 8- or 16-byte stores.  The block's threads are nh = min(H/4, 512) hidden-unit columns x
    // pgs pixel-group lanes: with one lane (the round-2 form, 128 threads for H = 512) a block walked its 49 pixel groups
    // one after the other, each a dependent chain of an L2 load and a short loop — 0.28 of the copy bandwidth
    // (profiles/r2_hbm_kernels.md); four lanes cut the chain to 13 and put 32 warps on an SM.
    const int nh = min(H >> 2, 512), pgs = max(1, (int)blockDim.x / nh);
    const int hg = threadIdx.x % nh, pg = threadIdx.x / nh;
    if (pg >= pgs) return;
    for (int h4 = hg * 4; h4 < H; h4 += nh * 4) {
      for (int p0 = pg * 4; p0 < P; p0 += pgs * 4) {
        float4 G[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const bool ok = p0 + k < P;
          const size_t o0 = ((size_t)b * P + (ok ? p0 + k : 0)) * H + h4;
          G[k] = ok ? __ldg(reinterpret_cast<const float4*>(w.gA + o0)) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
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
            for (int j = 0; j < 4; ++j) acc[k][j] = fmaf(al[k], uu[j], acc[k][j]);
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (p0 + k >= P) break;
          const size_t row = (size_t)q * P + p0 + k;
          const float g[4] = {G[k].x, G[k].y, G[k].z, G[k].w};
          if (SPLIT) {
            uint32_t hi2[2], lo2[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
              __nv_bfloat16 h0, l0, h1, l1;
              split_bf16(acc[k][2 * j] * g[2 * j], h0, l0);
              split_bf16(acc[k][2 * j + 1] * g[2 * j + 1], h1, l1);
              hi2[j] = (uint32_t)__bfloat16_as_ushort(h0) | ((uint32_t)__bfloat16_as_ushort(h1) << 16);
              lo2[j] = (uint32_t)__bfloat16_as_ushort(l0) | ((uint32_t)__bfloat16_as_ushort(l1) << 16);
            }
            __nv_bfloat16* o = w.a3 + row * 2 * H + h4;
            *reinterpret_cast<uint2*>(o) = make_uint2(hi2[0], hi2[1]);
            *reinterpret_cast<uint2*>(o + H) = make_uint2(lo2[0], lo2[1]);
          } else {
            *reinterpret_cast<float4*>(w.wproj + row * H + h4) =
                make_float4(acc[k][0] * g[0], acc[k][1] * g[1], acc[k][2] * g[2], acc[k][3] * g[3]);
          }
        }
      }
    }
    return;
  }
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    for (int p0 = 0; p0 < P; p0 += 4) {
      float Av[4], Ap[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const bool ok = p0 + k < P;
        const size_t o0 = ((size_t)b * P + (ok ? p0 + k : 0)) * H + h;
        Av[k] = ok ? __ldg(a.A + o0) : 0.f;
        Ap[k] = ok ? __ldg(a.A_pre + o0) : 1.f;
      }
      float acc[4] = {0.f, 0.f, 0.f, 0.f};
      for (int i = t; i >= 0; --i) {
        const float uv = u_s[i * H + h];
        const float4 a4 = *reinterpret_cast<const float4*>(al_s + i * P4 + p0);
        acc[0] = fmaf(a4.x, uv, acc[0]);
        acc[1] = fmaf(a4.y, uv, acc[1]);
        acc[2] = fmaf(a4.z, uv, acc[2]);
        acc[3] = fmaf(a4.w, uv, acc[3]);
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        if (p0 + k >= P) break;
        const size_t row = (size_t)q * P + p0 + k;
        if (SPLIT) {
          // the quotient is split into bf16 hi + lo (16 mantissa bits): the 2-ulp division is far below that
          const float r = __fdividef(acc[k] * Av[k], stab(Ap[k]));
          __nv_bfloat16 hi, lo;
          split_bf16(r, hi, lo);
          __nv_bfloat16* o = w.a3 + row * 2 * H;
          o[h] = hi; o[H + h] = lo;
        } else {
          w.wproj[row * H + h] = acc[k] * Av[k] / stab(Ap[k]);
        }
      }
    }
  }
}
static size_t grid_carve(const lrpx_gridtd_args* a, float* base, GridWs* w) {
  Carver c{base};
  size_t Q = a->Q, H = a->H, E = a->E;
  size_t nmax = 3 * H > 2 * H + 2 * E ? 3 * H : 2 * H + 2 * E;
  if ((size_t)a->C > nmax) nmax = a->C;
  GridWs t{};
  t.r_h2 = c.f32(Q * H); t.r_c2 = c.f32(Q * H); t.r_c1 = c.f32(Q * H); t.r_cth = c.f32(Q * H);
  t.r_glob = c.f32(Q * E);
  t.u = c.f32(Q * (H > E ? H : E));
  t.v = c.f32(Q * nmax);
  t.uctx = c.f32(Q * a->T * H);
  t.coefavg = c.f32(Q * a->C);
  t.wproj = c.f32(Q * a->P * H);
  t.gA = c.f32((size_t)a->B * a->P * H);
  if (a->flags & LRPX_DEC_TC_GEMM) {
    // a3: W_proj (Q*P, H), W_glob (Q, E), W_g2 and W_g1 (Q, H) unless fused;  a3u: W_g2 and W_g1 fused (Q, H)
    t.a3 = c.bf16(std::max({split_elems(Q * a->P, H), split_elems(Q, E), split_elems(Q, H)}));
    t.w3_g2 = c.bf16((size_t)3 * H * 3 * H);
    t.w3_g1 = c.bf16((size_t)(2 * H + 2 * E) * 3 * H);
    t.w3_glob = c.bf16((size_t)a->C * 3 * E);
    t.w3_proj = c.bf16((size_t)a->C * 3 * H);
    t.a3u = c.bf16(split_elems(Q, H));
  }
  if (w) *w = t;
  return c.bytes();
}

// ------------------------------------------------------------------------------------------------
// AoA
// ------------------------------------------------------------------------------------------------
struct AoaWs {
  float *r_h, *r_glob, *u, *v, *uval, *addq, *wval, *w2;
  __nv_bfloat16 *a3, *w3_aoa, *w3_g, *w3_v, *w3_proj;
};

__global__ void aoa_init_kernel(lrpx_aoa_args a, AoaWs w) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q], word = a.req_word[q];
  float logit = a.pred[((size_t)b * a.T + t) * a.V + word];
  float coef = logit / stab(logit);
  const float* h = a.h + ((size_t)b * (a.T + 1) + t + 1) * a.H;
  const float* ca = a.caoa + ((size_t)b * a.T + t) * a.H;
  const float* cl = a.caoa_lin + ((size_t)b * a.T + t) * a.H;
  const float* wr = a.W_fc + (size_t)word * a.H;
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    float rh, rc;
    fc_split(h[j], ca[j], wr[j], coef, rh, rc);               // :1092-1104
    w.r_h[(size_t)q * a.H + j] = rh;
    w.u[(size_t)q * a.H + j] = rc / stab(cl[j]);              // lin() through decoder_aoa_linear (:1107-1110)
    w.r_glob[(size_t)q * a.H + j] = 0.f;
  }
  zero_words(a, q);
}
// r_ctx = ctx * v ;  uval = r_ctx / stab(ctx) on the chosen head, 0 elsewhere (lrp_mha :848-860, Q5)
__global__ void aoa_ctx_kernel(lrpx_aoa_args a, AoaWs w) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q], head = a.req_head[q];
  int dk = a.H / a.num_head;
  const float* cx = a.ctx + ((size_t)b * a.T + t) * a.H;
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    float r_ctx = cx[j] * w.v[(size_t)q * a.H + j];
    w.uval[(size_t)q * a.H + j] = (j / dk == head) ? r_ctx / stab(cx[j]) : 0.f;
  }
}
// LSTM chain without cell carry (Q4, :1115-1124): r_g = ident(r_h[i+1], i*tanh(g), c[i+1])
__global__ void aoa_cell_kernel(lrpx_aoa_args a, AoaWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  bool active = i <= t;
  size_t bi = ((size_t)b * a.T + i) * a.H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * a.H;
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    size_t o = (size_t)q * a.H + j;
    if (!active) { w.u[o] = 0.f; continue; }
    float g = a.g[bi + j];
    float r_g = a.i[bi + j] * tanhf(g) * w.r_h[o] / stab(a.c[bi1 + j]);
    w.u[o] = r_g / stab(g);
  }
}
__global__ void aoa_post_kernel(lrpx_aoa_args a, AoaWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  if (i > t) return;
  const int H = a.H, E = a.E;
  const float* x = a.x + ((size_t)b * a.T + i) * (E + H);
  const float* hh = a.h + ((size_t)b * (a.T + 1) + i) * H;
  const float* vq = w.v + (size_t)q * (E + 2 * H);
  float wsum = 0.f;
  for (int k = threadIdx.x; k < E + 2 * H; k += blockDim.x) {
    float xv = k < E + H ? x[k] : hh[k - E - H];
    float rx = xv * vq[k];
    if (k < E) wsum += rx;                                            // :1130
    else if (k < E + H) w.r_glob[(size_t)q * H + (k - E)] += rx;      // :1133
    else w.r_h[(size_t)q * H + (k - E - H)] = rx;                     // :1129
  }
  block_sum_store(wsum, [&](float s) { store_word(a, q, i, s); });
}
// wval = r_val / stab(value), r_val = value * alpha[head][p] * uval   (:1112-1113, :1141-1144)
// addq = r_glob / stab(glob) / P                                     (:1136-1139)
__global__ void aoa_val_kernel(lrpx_aoa_args a, AoaWs w) {
  const int q = blockIdx.x / a.P, p = blockIdx.x - q * a.P;          // one block per (request, pixel)
  int b = a.req_img[q], t = a.req_t[q], head = a.req_head[q];
  float al = a.alpha[(((size_t)b * a.T + t) * a.num_head + head) * a.P + p];
  size_t o0 = ((size_t)b * a.P + p) * a.H;
  for (int h = threadIdx.x; h < a.H; h += blockDim.x) {
    float val = a.value[o0 + h];
    w.wval[((size_t)q * a.P + p) * a.H + h] = val * al * w.uval[(size_t)q * a.H + h] / stab(val);
    if (p == 0) w.addq[(size_t)q * a.H + h] = w.r_glob[(size_t)q * a.H + h] / stab(a.glob[(size_t)b * a.H + h]) / (float)a.P;
  }
}

static size_t aoa_carve(const lrpx_aoa_args* a, float* base, AoaWs* w) {
  Carver c{base};
  size_t Q = a->Q, H = a->H;
  AoaWs t{};
  t.r_h = c.f32(Q * H); t.r_glob = c.f32(Q * H); t.u = c.f32(Q * H);
  t.v = c.f32(Q * (a->E + 2 * H));
  t.uval = c.f32(Q * H); t.addq = c.f32(Q * H);
  t.wval = c.f32(Q * a->P * H);
  t.w2 = c.f32(Q * a->P * H);
  if (a->flags & LRPX_DEC_TC_GEMM) {
    // a3: W_v and W_proj (Q*P, H), W_aoa and W_g (Q, H)
    t.a3 = c.bf16(std::max(split_elems(Q * a->P, H), split_elems(Q, H)));
    t.w3_aoa = c.bf16(H * 3 * H);
    t.w3_g = c.bf16((size_t)(a->E + 2 * H) * 3 * H);
    t.w3_v = c.bf16(H * 3 * H);
    t.w3_proj = c.bf16((size_t)a->C * 3 * H);
  }
  if (w) *w = t;
  return c.bytes();
}

// ------------------------------------------------------------------------------------------------
// Adaptive attention (single AdaLSTM): ExplainAdaptiveAttention.explain_caption_wordt, adaptiveattention.py:679-771
// ------------------------------------------------------------------------------------------------
struct AdaWs {
  float *r_h, *r_c, *r_glob, *u, *v, *uctx, *coefavg, *wproj;
  __nv_bfloat16 *a3, *w3_g, *w3_glob, *w3_proj;
  __nv_bfloat16* a3u;      // split form of u written by the cell kernel itself (null: CUDA-core GEMM)
};

// fc rule on the target row, split into h / ctx_hat, ctx_hat into context / sentinel (:700-724)
__global__ void ada_init_kernel(lrpx_adaptive_args a, AdaWs w) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q], word = a.req_word[q];
  float logit = a.pred[((size_t)b * a.T + t) * a.V + word];
  float coef = logit / stab(logit);
  const float* h = a.h + ((size_t)b * (a.T + 1) + t + 1) * a.H;
  size_t bi = ((size_t)b * a.T + t) * a.H;
  const float* wr = a.W_fc + (size_t)word * a.H;
  float beta = a.beta[(size_t)b * a.T + t];
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    float rh, rcth;
    float cth = a.ctx_hat[bi + j];
    fc_split(h[j], cth, wr[j], coef, rh, rcth);
    float dct = stab(cth);
    float cx = a.ctx[bi + j];
    float r_ctx = (1.f - beta) * cx * rcth / dct;
    size_t o = (size_t)q * a.H + j;
    w.r_h[o] = rh;
    w.r_c[o] = beta * a.st[bi + j] * rcth / dct;          // r_ct[t+1] = r_st (:724)
    w.uctx[o] = r_ctx / stab(cx);
  }
  for (int j = threadIdx.x; j < a.E; j += blockDim.x) w.r_glob[(size_t)q * a.E + j] = 0.f;
  zero_words(a, q);
}

// cell rule (:726-734) -> u = r_g / stab(tanh g)   (the reference passes tanh(gt) as forward_output, :737)
__global__ void ada_cell_kernel(lrpx_adaptive_args a, AdaWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  bool active = i <= t;
  size_t bi = ((size_t)b * a.T + i) * a.H, bi1 = ((size_t)b * (a.T + 1) + i + 1) * a.H,
         bi0 = ((size_t)b * (a.T + 1) + i) * a.H;
  for (int j = threadIdx.x; j < a.H; j += blockDim.x) {
    size_t o = (size_t)q * a.H + j;
    if (!active) { put_operand(w.u, w.a3u, q, a.H, j, 0.f); continue; }
    float rc = w.r_c[o] + w.r_h[o];
    float d = stab(a.c[bi1 + j]);
    float tg = tanhf(a.g[bi + j]);
    float r_g = a.i[bi + j] * tg * rc / d;
    w.r_c[o] = a.f[bi + j] * a.c[bi0 + j] * rc / d;
    put_operand(w.u, w.a3u, q, a.H, j, r_g / stab(tg));
  }
}

// after v = u @ W_g : slices of xht = [emb | glob | h_i] (:739-742)
__global__ void ada_post_kernel(lrpx_adaptive_args a, AdaWs w, int i) {
  int q = blockIdx.x;
  int b = a.req_img[q], t = a.req_t[q];
  if (i > t) return;
  const int H = a.H, E = a.E;
  const float* x = a.x + ((size_t)b * a.T + i) * 2 * E;
  const float* hp = a.h + ((size_t)b * (a.T + 1) + i) * H;
  const float* vq = w.v + (size_t)q * (2 * E + H);
  float wsum = 0.f;
  for (int k = threadIdx.x; k < 2 * E + H; k += blockDim.x) {
    if (k < E) wsum += x[k] * vq[k];
    else if (k < 2 * E) { if (i == t) w.r_glob[(size_t)q * E + (k - E)] = x[k] * vq[k]; }   // only the explained step (:740)
    else w.r_h[(size_t)q * H + (k - 2 * E)] = hp[k - 2 * E] * vq[k];
  }
  block_sum_store(wsum, [&](float s) { store_word(a, q, i, s); });
}

// u_g = r_glob / stab(avg @ W_glob^T)   (:743-746, forward_output=False: no bias)
__global__ void ada_glob_kernel(lrpx_adaptive_args a, AdaWs w) {
  int q = blockIdx.x, b = a.req_img[q];
  for (int j = threadIdx.x; j < a.E; j += blockDim.x)
    w.u[(size_t)q * a.E + j] = w.r_glob[(size_t)q * a.E + j] / stab(a.z_glob[(size_t)b * a.E + j]);
}
// coefavg = avg * v / stab(avg) / P  (mean rule :752-755 applied to r_avg = avg * v)
__global__ void ada_avg_kernel(lrpx_adaptive_args a, AdaWs w) {
  int q = blockIdx.x, b = a.req_img[q];
  for (int c = threadIdx.x; c < a.C; c += blockDim.x) {
    float av = a.avg[(size_t)b * a.C + c];
    float r_avg = av * w.v[(size_t)q * a.C + c];
    w.coefavg[(size_t)q * a.C + c] = r_avg / stab(av) / (float)a.P;
  }
}
// attention weighted-sum rule at the explained step only (:756-759), already divided for the projector rule (:760-763):
//   wproj[q][p][h] = A[p][h] * alpha_t[p] * uctx[h] / stab(z_proj[p][h]);  block = (request, pixel group of 8)
template <bool SPLIT>
__global__ void __launch_bounds__(256) ada_attn_kernel(lrpx_adaptive_args a, AdaWs w) {
  const int H = a.H, P = a.P;
  const int ng = (P + 7) / 8;
  const int q = blockIdx.x / ng;
  const int b = a.req_img[q], t = a.req_t[q];
  const int p0 = (blockIdx.x - q * ng) * 8, p1 = min(P, p0 + 8);
  const float* al = a.alpha + ((size_t)b * a.T + t) * P;
  for (int h = threadIdx.x; h < H; h += blockDim.x) {
    const float uv = w.uctx[(size_t)q * H + h];
    for (int p = p0; p < p1; ++p) {
      const size_t o0 = ((size_t)b * P + p) * H + h;
      const size_t row = (size_t)q * P + p;
      const float num = __ldg(a.A + o0) * al[p] * uv, den = stab(__ldg(a.z_proj + o0));
      if (SPLIT) {
        __nv_bfloat16 hi, lo;
        split_bf16(__fdividef(num, den), hi, lo);       // bf16 hi + lo keeps 16 mantissa bits: above the 2-ulp division
        __nv_bfloat16* o = w.a3 + row * 2 * H;
        o[h] = hi; o[H + h] = lo;
      } else {
        w.wproj[row * H + h] = num / den;
      }
    }
  }
}

static size_t ada_carve(const lrpx_adaptive_args* a, float* base, AdaWs* w) {
  Carver c{base};
  size_t Q = a->Q, H = a->H, E = a->E;
  size_t nmax = 2 * E + H > (size_t)a->C ? 2 * E + H : (size_t)a->C;
  AdaWs t{};
  t.r_h = c.f32(Q * H); t.r_c = c.f32(Q * H);
  t.r_glob = c.f32(Q * E);
  t.u = c.f32(Q * (H > E ? H : E));
  t.v = c.f32(Q * nmax);
  t.uctx = c.f32(Q * H);
  t.coefavg = c.f32(Q * a->C);
  t.wproj = c.f32(Q * a->P * H);
  if (a->flags & LRPX_DEC_TC_GEMM) {
    // a3: W_proj (Q*P, H), W_glob (Q, E);  a3u: W_g, always fused (Q, H)
    t.a3 = c.bf16(std::max(split_elems(Q * a->P, H), split_elems(Q, E)));
    t.w3_g = c.bf16((size_t)(2 * E + H) * 3 * H);
    t.w3_glob = c.bf16((size_t)a->C * 3 * E);
    t.w3_proj = c.bf16((size_t)a->C * 3 * H);
    t.a3u = c.bf16(split_elems(Q, H));
  }
  if (w) *w = t;
  return c.bytes();
}

// ------------------------------------------------------------------------------------------------
// lrp_tune weights: one block per sample
// ------------------------------------------------------------------------------------------------
__global__ void fc_lrp_weights_kernel(const float* __restrict__ logits, const float* __restrict__ h,
                                      const float* __restrict__ ctx, const float* __restrict__ W_fc,
                                      const uint8_t* __restrict__ is_stop, float* __restrict__ w_ctx,
                                      float* __restrict__ w_h, int32_t* __restrict__ argmax_out, int V, int H) {
  int b = blockIdx.x;
  const float* lg = logits + (size_t)b * V;
  __shared__ float s_val[32];
  __shared__ int s_idx[32];
  __shared__ float s_m[2][32];
  // argmax, first index wins on ties (torch.argmax, gridTDmodel.py:555); NaN counts as the maximum (torch's order:
  // a diverged tuning run with NaN logits returns the first NaN's index there and must not index out of bounds here)
  auto better = [](float v, int j, float bv, int bi) {
    const bool vn = v != v, bn = bv != bv;
    if (vn || bn) return vn && (!bn || j < bi);
    return v > bv || (v == bv && j < bi);
  };
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int j = threadIdx.x; j < V; j += blockDim.x) {
    float v = lg[j];
    if (better(v, j, bv, bi)) { bv = v; bi = j; }
  }
  for (int o = 16; o; o >>= 1) {
    float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
  }
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) / 32;
  if (lane == 0) { s_val[wid] = bv; s_idx[wid] = bi; }
  __syncthreads();
  if (wid == 0) {
    bv = lane < nw ? s_val[lane] : -INFINITY;
    bi = lane < nw ? s_idx[lane] : 0x7fffffff;
    for (int o = 16; o; o >>= 1) {
      float ov = __shfl_xor_sync(0xffffffffu, bv, o);
      int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (better(ov, oi, bv, bi)) { bv = ov; bi = oi; }
    }
    if (lane == 0) { s_val[0] = bv; s_idx[0] = (bi >= 0 && bi < V) ? bi : 0; }
  }
  __syncthreads();
  int word = s_idx[0];
  float logit = s_val[0];
  if (argmax_out && threadIdx.x == 0) argmax_out[b] = word;
  bool stop = is_stop[word] != 0;                                   // Q15
  float coef = logit / stab(logit);
  const float* wr = W_fc + (size_t)word * H;
  // pass 1: max |r|
  float mh = 0.f, mc = 0.f;
  if (!stop)
    for (int j = threadIdx.x; j < H; j += blockDim.x) {
      float rh, rc;
      fc_split(h[(size_t)b * H + j], ctx[(size_t)b * H + j], wr[j], coef, rh, rc);
      mh = fmaxf(mh, fabsf(rh));
      mc = fmaxf(mc, fabsf(rc));
    }
  for (int o = 16; o; o >>= 1) {
    mh = fmaxf(mh, __shfl_xor_sync(0xffffffffu, mh, o));
    mc = fmaxf(mc, __shfl_xor_sync(0xffffffffu, mc, o));
  }
  if (lane == 0) { s_m[0][wid] = mh; s_m[1][wid] = mc; }
  __syncthreads();
  mh = 0.f; mc = 0.f;
  for (int k = 0; k < nw; ++k) { mh = fmaxf(mh, s_m[0][k]); mc = fmaxf(mc, s_m[1][k]); }
  if (mh == 0.f) mh = 1.f;                                          // utils.py:59
  if (mc == 0.f) mc = 1.f;
  for (int j = threadIdx.x; j < H; j += blockDim.x) {
    float rh = 0.f, rc = 0.f;
    if (!stop) fc_split(h[(size_t)b * H + j], ctx[(size_t)b * H + j], wr[j], coef, rh, rc);
    w_h[(size_t)b * H + j] = rh / mh + 1.f;
    w_ctx[(size_t)b * H + j] = rc / mc + 1.f;
  }
}

}  // namespace lrpx

using namespace lrpx;

extern "C" {

size_t lrpx_gridtd_decoder_workspace_bytes(const lrpx_gridtd_args* a) {
  if (!a) return 0;
  return grid_carve(a, nullptr, nullptr);
}

int lrpx_gridtd_decoder_lrp_f32(const lrpx_gridtd_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->B > 0 && a->T > 0 && a->H > 0 && a->E > 0 && a->P > 0 && a->C > 0 && a->V > 0 && a->Q >= 0,
                 "bad dimensions");
  if (a->Q == 0) return LRPX_OK;
  LRPX_CHECK_ARG(a->feat && a->avg && a->A_pre && a->A && a->glob_pre && a->x1 && a->x2 && a->h1 && a->c1 && a->h2 &&
                     a->c2 && a->g1 && a->i1 && a->f1 && a->g2 && a->i2 && a->f2 && a->st && a->ctx && a->ctx_hat &&
                     a->alpha && a->beta && a->pred && a->W_g1 && a->W_g2 && a->W_fc && a->W_glob && a->W_proj &&
                     a->req_img && a->req_t && a->req_word && a->r_feat && a->r_words,
                 "null pointer in args");
  GridWs w;
  size_t need = grid_carve(a, (float*)workspace, &w);
  LRPX_CHECK_ARG(workspace && workspace_bytes >= need, "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Q = a->Q, H = a->H, E = a->E, T = a->T;
  int nt = H >= 256 ? 256 : 128;
  GemmEpi none{};
  // tensor-core GEMMs where the shape allows it (per GEMM), CUDA cores otherwise
  const bool tc = (a->flags & LRPX_DEC_TC_GEMM) != 0;
  const bool w3_ready = (a->flags & LRPX_DEC_W3_READY) != 0;
  const __nv_bfloat16* w3_g2 = tc_weight(tc, a->W_g2, w.w3_g2, H, 3 * H, st, w3_ready);
  const __nv_bfloat16* w3_g1 = tc_weight(tc, a->W_g1, w.w3_g1, H, 2 * H + 2 * E, st, w3_ready);
  const __nv_bfloat16* w3_glob = tc_weight(tc, a->W_glob, w.w3_glob, E, a->C, st, w3_ready);
  const __nv_bfloat16* w3_proj = tc_weight(tc, a->W_proj, w.w3_proj, H, a->C, st, w3_ready);
  // the step kernels write the split operand themselves when both step GEMMs run on the tensor cores
  const bool fused_split = w3_g2 && w3_g1;
  if (!fused_split) w.a3u = nullptr;
  __nv_bfloat16* a3_step = fused_split ? w.a3u : w.a3;
  grid_init_kernel<<<Q, nt, 0, st>>>(*a, w);
  cudaMemsetAsync(w.uctx, 0, (size_t)Q * T * H * sizeof(float), st);
  for (int i = T - 1; i >= 0; --i) {
    grid_cell2_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W_g2, w3_g2, a3_step, w.v, Q, 3 * H, H, none, st, fused_split));
    grid_post2_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W_g1, w3_g1, a3_step, w.v, Q, 2 * H + 2 * E, H, none, st, fused_split));
    grid_post1_kernel<<<Q, 256, 0, st>>>(*a, w, i);
  }
  grid_glob_kernel<<<Q, 128, 0, st>>>(*a, w);
  RUN(gemm_any<GE_STORE>(w.u, a->W_glob, w3_glob, w.a3, w.v, Q, a->C, E, none, st));
  grid_avg_kernel<<<Q, 128, 0, st>>>(*a, w);
  GemmEpi fe{a->feat, nullptr, w.coefavg, a->req_img, a->P};
  const size_t att_smem = (size_t)T * (((a->P + 3) & ~3) + H) * sizeof(float);
  if (att_smem <= 160 * 1024) {
    int at = H >= 512 ? 512 : (H >= 256 ? 256 : 128);
    if ((H & 3) == 0) {                  // four hidden units per thread x as many pixel-group lanes as fit 512 threads
      const int nh = H / 4 >= 512 ? 512 : H / 4;
      at = (nh * (512 / nh > 0 ? 512 / nh : 1) + 31) & ~31;
      const size_t n4 = (size_t)a->B * a->P * H / 4;
      grid_attn_gain_kernel<<<(unsigned)((n4 + 255) / 256 < 4096 ? (n4 + 255) / 256 : 4096), 256, 0, st>>>(a->A, a->A_pre, w.gA, n4);
    }
    static std::atomic<uint64_t> attr_done[2];
    if (w3_proj) {
      RUN(ensure_smem_attr(grid_attn_rows_kernel<true>, 160 * 1024, attr_done[1]));
      grid_attn_rows_kernel<true><<<Q, at, att_smem, st>>>(*a, w);
    } else {
      RUN(ensure_smem_attr(grid_attn_rows_kernel<false>, 160 * 1024, attr_done[0]));
      grid_attn_rows_kernel<false><<<Q, at, att_smem, st>>>(*a, w);
    }
    RUN(gemm_any<GE_FEAT>(w.wproj, a->W_proj, w3_proj, w.a3, a->r_feat, Q * a->P, a->C, H, fe, st, w3_proj != nullptr));
  } else {
    grid_attn_kernel<<<(unsigned)Q * a->P, nt, 0, st>>>(*a, w);
    RUN(gemm_any<GE_FEAT>(w.wproj, a->W_proj, w3_proj, w.a3, a->r_feat, Q * a->P, a->C, H, fe, st));
  }
  words_norm_kernel<<<Q, 32, 0, st>>>(a->r_words, a->req_t, T);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

size_t lrpx_aoa_decoder_workspace_bytes(const lrpx_aoa_args* a) {
  if (!a) return 0;
  return aoa_carve(a, nullptr, nullptr);
}

int lrpx_aoa_decoder_lrp_f32(const lrpx_aoa_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->B > 0 && a->T > 0 && a->H > 0 && a->E > 0 && a->P > 0 && a->C > 0 && a->V > 0 && a->Q >= 0 &&
                     a->num_head > 0 && a->H % a->num_head == 0,
                 "bad dimensions");
  if (a->Q == 0) return LRPX_OK;
  LRPX_CHECK_ARG(a->feat && a->A_pre && a->A && a->glob && a->value && a->x && a->h && a->c && a->g && a->i &&
                     a->ctx && a->caoa && a->caoa_lin && a->alpha && a->pred && a->W_g && a->W_fc && a->W_aoa &&
                     a->W_v && a->W_proj && a->req_img && a->req_t && a->req_word && a->req_head && a->r_feat &&
                     a->r_words,
                 "null pointer in args");
  AoaWs w;
  size_t need = aoa_carve(a, (float*)workspace, &w);
  LRPX_CHECK_ARG(workspace && workspace_bytes >= need, "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Q = a->Q, H = a->H, E = a->E, T = a->T;
  int nt = H >= 256 ? 256 : 128;
  GemmEpi none{};
  const bool tc = (a->flags & LRPX_DEC_TC_GEMM) != 0;
  const bool w3_ready = (a->flags & LRPX_DEC_W3_READY) != 0;
  const __nv_bfloat16* w3_aoa = tc_weight(tc, a->W_aoa, w.w3_aoa, H, H, st, w3_ready);
  const __nv_bfloat16* w3_g = tc_weight(tc, a->W_g, w.w3_g, H, E + 2 * H, st, w3_ready);
  const __nv_bfloat16* w3_v = tc_weight(tc, a->W_v, w.w3_v, H, H, st, w3_ready);
  const __nv_bfloat16* w3_proj = tc_weight(tc, a->W_proj, w.w3_proj, H, a->C, st, w3_ready);
  aoa_init_kernel<<<Q, nt, 0, st>>>(*a, w);
  RUN(gemm_any<GE_STORE>(w.u, a->W_aoa, w3_aoa, w.a3, w.v, Q, H, H, none, st));
  aoa_ctx_kernel<<<Q, nt, 0, st>>>(*a, w);
  for (int i = T - 1; i >= 0; --i) {
    aoa_cell_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W_g, w3_g, w.a3, w.v, Q, E + 2 * H, H, none, st));
    aoa_post_kernel<<<Q, 256, 0, st>>>(*a, w, i);
  }
  aoa_val_kernel<<<(unsigned)Q * a->P, nt, 0, st>>>(*a, w);
  GemmEpi pe{a->A, a->A_pre, w.addq, a->req_img, a->P};
  RUN(gemm_any<GE_AOA_PROJ>(w.wval, a->W_v, w3_v, w.a3, w.w2, Q * a->P, H, H, pe, st));
  GemmEpi fe{a->feat, nullptr, nullptr, a->req_img, a->P};
  RUN(gemm_any<GE_FEAT>(w.w2, a->W_proj, w3_proj, w.a3, a->r_feat, Q * a->P, a->C, H, fe, st));
  words_norm_kernel<<<Q, 32, 0, st>>>(a->r_words, a->req_t, T);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

size_t lrpx_adaptive_decoder_workspace_bytes(const lrpx_adaptive_args* a) {
  if (!a) return 0;
  return ada_carve(a, nullptr, nullptr);
}

int lrpx_adaptive_decoder_lrp_f32(const lrpx_adaptive_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->B > 0 && a->T > 0 && a->H > 0 && a->E > 0 && a->P > 0 && a->C > 0 && a->V > 0 && a->Q >= 0,
                 "bad dimensions");
  if (a->Q == 0) return LRPX_OK;
  LRPX_CHECK_ARG(a->feat && a->avg && a->z_proj && a->A && a->z_glob && a->x && a->h && a->c && a->g && a->i && a->f &&
                     a->st && a->ctx && a->ctx_hat && a->alpha && a->beta && a->pred && a->W_g && a->W_fc && a->W_glob &&
                     a->W_proj && a->req_img && a->req_t && a->req_word && a->r_feat && a->r_words,
                 "null pointer in args");
  AdaWs w;
  size_t need = ada_carve(a, (float*)workspace, &w);
  LRPX_CHECK_ARG(workspace && workspace_bytes >= need, "workspace too small");
  cudaStream_t st = as_stream(stream);
  const int Q = a->Q, H = a->H, E = a->E, T = a->T;
  int nt = H >= 256 ? 256 : 128;
  GemmEpi none{};
  const bool tc = (a->flags & LRPX_DEC_TC_GEMM) != 0;
  const bool w3_ready = (a->flags & LRPX_DEC_W3_READY) != 0;
  const __nv_bfloat16* w3_g = tc_weight(tc, a->W_g, w.w3_g, H, 2 * E + H, st, w3_ready);
  const __nv_bfloat16* w3_glob = tc_weight(tc, a->W_glob, w.w3_glob, E, a->C, st, w3_ready);
  const __nv_bfloat16* w3_proj = tc_weight(tc, a->W_proj, w.w3_proj, H, a->C, st, w3_ready);
  if (!w3_g) w.a3u = nullptr;
  ada_init_kernel<<<Q, nt, 0, st>>>(*a, w);
  for (int i = T - 1; i >= 0; --i) {
    ada_cell_kernel<<<Q, nt, 0, st>>>(*a, w, i);
    RUN(gemm_any<GE_STORE>(w.u, a->W_g, w3_g, w.a3u, w.v, Q, 2 * E + H, H, none, st, w3_g != nullptr));
    ada_post_kernel<<<Q, 256, 0, st>>>(*a, w, i);
  }
  ada_glob_kernel<<<Q, 128, 0, st>>>(*a, w);
  RUN(gemm_any<GE_STORE>(w.u, a->W_glob, w3_glob, w.a3, w.v, Q, a->C, E, none, st));
  ada_avg_kernel<<<Q, 128, 0, st>>>(*a, w);
  GemmEpi fe{a->feat, nullptr, w.coefavg, a->req_img, a->P};
  const unsigned ag = (unsigned)((a->P + 7) / 8) * (unsigned)Q;
  if (w3_proj) ada_attn_kernel<true><<<ag, nt, 0, st>>>(*a, w);
  else ada_attn_kernel<false><<<ag, nt, 0, st>>>(*a, w);
  RUN(gemm_any<GE_FEAT>(w.wproj, a->W_proj, w3_proj, w.a3, a->r_feat, Q * a->P, a->C, H, fe, st, w3_proj != nullptr));
  words_norm_kernel<<<Q, 32, 0, st>>>(a->r_words, a->req_t, T);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_fc_lrp_weights_f32(const float* logits, const float* h, const float* ctx, const float* W_fc,
                            const uint8_t* is_stop, float* w_ctx, float* w_h, int32_t* argmax_out, int B, int V, int H,
                            void* stream) {
  LRPX_CHECK_ARG(logits && h && ctx && W_fc && is_stop && w_ctx && w_h && B >= 0 && V > 0 && H > 0, "bad argument");
  if (B == 0) return LRPX_OK;
  fc_lrp_weights_kernel<<<B, 256, 0, as_stream(stream)>>>(logits, h, ctx, W_fc, is_stop, w_ctx, w_h, argmax_out, V, H);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

}  // extern "C"
