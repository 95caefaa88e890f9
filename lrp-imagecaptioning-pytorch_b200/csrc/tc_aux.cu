// Helpers of the tensor-core path: weight preparation, the cin=3 first layer, 2x2 max-pool with argmax and
// gain gather, chain entry scaling and PF <-> dense conversions.  All HBM-bound, 16-byte vector accesses.
// PF layout: see include/lrpx.h ("padded-flat NHWC bf16").
#include "lrpx_common.cuh"
#include <cuda_fp16.h>

namespace lrpx {

static inline int grid_for(long long total, int block = 256) {
  long long g = (total + block - 1) / block, cap = 148LL * 16;
  return (int)(g < 1 ? 1 : (g > cap ? cap : g));
}

// fp32 (cout,cin,kh,kw) -> bf16 GEMM operand, see lrpx_weight_prep_bf16 in lrpx.h
__global__ void weight_prep_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ wt, int cout, int cin,
                                   int kh, int kw, int mode, int rows_pad, int chan_pad) {
  long long total = (long long)rows_pad * kh * kw * chan_pad;
  bool transposed = mode >= 2;
  int rows = transposed ? cin : cout, chans = transposed ? cout : cin;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int c = (int)(i % chan_pad);
    int rs = (int)((i / chan_pad) % (kh * kw));
    int row = (int)(i / ((long long)chan_pad * kh * kw));
    float v = 0.f;
    if (row < rows && c < chans) {
      int r = rs / kw, s = rs % kw;
      if (!transposed) {
        v = w[(((size_t)row * cin + c) * kh + r) * kw + s];
        if (mode == 1) v = fmaxf(v, 0.f);
      } else {
        v = w[(((size_t)c * cin + row) * kh + (kh - 1 - r)) * kw + (kw - 1 - s)];
        v = (mode == 2) ? fmaxf(v, 0.f) : fminf(v, 0.f);
      }
    }
    wt[i] = __float2bfloat16(v);
  }
}

// ---------------------------------------------------------------- first layer (cin = 3), CUDA cores
// One thread = FF_PX consecutive PF rows x 8 output channels; a warp = 4 row groups x 8 channel groups (cout = 64), so
// every store instruction writes 4 full 128-byte PF rows.  Shared memory holds W, W+ and W- in the order
// [array][tap][quad][channel group][4] — the 8 channel groups of a warp read 128 contiguous bytes per LDS.128, and a
// weight fetched once feeds FF_PX pixels (with one pixel per thread and a [tap][cout] layout the kernel was bound by
// shared-memory bandwidth: 2-way bank conflicts on every LDS.128, 3.7 ms for 64 images).  One (tap, channel pair)
// costs three packed fma.rn.f32x2: z += w*x, z+ += w+*x+, z+ += w-*x-  (lrp_modules.py:81-84, mixed-sign input).
constexpr int FF_PX = 4;
template <int CG>   // channel groups per pixel = cout / 8
__global__ void __launch_bounds__(256) first_fwd_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                        const float* __restrict__ bias, uint4* __restrict__ act,
                                                        uint4* __restrict__ gain, int n, int h, int wd) {
  extern __shared__ __align__(16) float ws[];        // [3][27][2][CG][4] (w, w+, w-), then bias[cout]
  constexpr int cout = CG * 8;
  for (int i = threadIdx.x; i < 27 * cout; i += blockDim.x) {
    const int k = i / cout, co = i % cout;           // k = (ci, r, s) of (cout,3,3,3)
    const int cg = co >> 3, q = (co >> 2) & 1, e = co & 3;
    const float v = w[co * 27 + k];
    const int o = ((k * 2 + q) * CG + cg) * 4 + e;
    ws[o] = v;
    ws[27 * cout + o] = fmaxf(v, 0.f);
    ws[2 * 27 * cout + o] = fminf(v, 0.f);
  }
  for (int i = threadIdx.x; i < cout; i += blockDim.x) ws[3 * 27 * cout + i] = bias ? bias[i] : 0.f;
  __syncthreads();
  const int wp1 = wd + 1, blk = (h + 1) * wp1;
  const long long rows = (long long)n * blk;
  const long long groups = (rows + FF_PX - 1) / FF_PX;
  const long long total = groups * CG;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % CG);
    const long long prow0 = (i / CG) * FF_PX;
    const float* xb[FF_PX];      // image base of each pixel (nullptr: padding row or past the end)
    int py[FF_PX], pxx[FF_PX];
#pragma unroll
    for (int j = 0; j < FF_PX; ++j) {
      const long long prow = prow0 + j;
      const int img = (int)(prow / blk), rem = (int)(prow % blk);
      const int a = rem / wp1, b = rem % wp1;
      const bool valid = prow < rows && a > 0 && b > 0;
      xb[j] = valid ? x + (size_t)img * 3 * h * wd : nullptr;
      py[j] = a - 1;
      pxx[j] = b - 1;
    }
    float2 z[FF_PX][4], zp[FF_PX][4];
#pragma unroll
    for (int j = 0; j < FF_PX; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        z[j][c] = make_float2(ws[3 * 27 * cout + cg * 8 + 2 * c], ws[3 * 27 * cout + cg * 8 + 2 * c + 1]);
        zp[j][c] = make_float2(0.f, 0.f);
      }
#pragma unroll
    for (int ci = 0; ci < 3; ++ci)
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int s = 0; s < 3; ++s) {
          const int k = (ci * 3 + r) * 3 + s;
          float4 wv[2], pv[2], nv[2];
#pragma unroll
          for (int q = 0; q < 2; ++q) {
            wv[q] = *reinterpret_cast<const float4*>(ws + ((k * 2 + q) * CG + cg) * 4);
            pv[q] = *reinterpret_cast<const float4*>(ws + 27 * cout + ((k * 2 + q) * CG + cg) * 4);
            nv[q] = *reinterpret_cast<const float4*>(ws + 2 * 27 * cout + ((k * 2 + q) * CG + cg) * 4);
          }
#pragma unroll
          for (int j = 0; j < FF_PX; ++j) {
            const int yy = py[j] + r - 1, xs = pxx[j] + s - 1;
            float xv = 0.f;
            if (xb[j] && yy >= 0 && yy < h && xs >= 0 && xs < wd) xv = __ldg(xb[j] + ((size_t)ci * h + yy) * wd + xs);
            const float2 x2 = make_float2(xv, xv);
            const float2 xp2 = make_float2(fmaxf(xv, 0.f), fmaxf(xv, 0.f));
            const float2 xn2 = make_float2(fminf(xv, 0.f), fminf(xv, 0.f));
#pragma unroll
            for (int q = 0; q < 2; ++q) {
              z[j][2 * q] = __ffma2_rn(make_float2(wv[q].x, wv[q].y), x2, z[j][2 * q]);
              z[j][2 * q + 1] = __ffma2_rn(make_float2(wv[q].z, wv[q].w), x2, z[j][2 * q + 1]);
              zp[j][2 * q] = __ffma2_rn(make_float2(pv[q].x, pv[q].y), xp2, zp[j][2 * q]);
              zp[j][2 * q + 1] = __ffma2_rn(make_float2(pv[q].z, pv[q].w), xp2, zp[j][2 * q + 1]);
              zp[j][2 * q] = __ffma2_rn(make_float2(nv[q].x, nv[q].y), xn2, zp[j][2 * q]);
              zp[j][2 * q + 1] = __ffma2_rn(make_float2(nv[q].z, nv[q].w), xn2, zp[j][2 * q + 1]);
            }
          }
        }
#pragma unroll
    for (int j = 0; j < FF_PX; ++j) {
      if (prow0 + j >= rows) break;
      uint4 oa = make_uint4(0, 0, 0, 0), og = make_uint4(0, 0, 0, 0);
      if (xb[j]) {
        uint32_t pa[4], pg[4];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          float a0 = fmaxf(z[j][c].x, 0.f), a1 = fmaxf(z[j][c].y, 0.f);
          __nv_bfloat162 ta = __floats2bfloat162_rn(a0, a1);
          __nv_bfloat162 tg = __floats2bfloat162_rn(safe_div(a0, zp[j][c].x), safe_div(a1, zp[j][c].y));
          pa[c] = *reinterpret_cast<uint32_t*>(&ta);
          pg[c] = *reinterpret_cast<uint32_t*>(&tg);
        }
        oa = make_uint4(pa[0], pa[1], pa[2], pa[3]);
        og = make_uint4(pg[0], pg[1], pg[2], pg[3]);
      }
      act[(prow0 + j) * CG + cg] = oa;
      gain[(prow0 + j) * CG + cg] = og;
    }
  }
}

// ---------------------------------------------------------------- 2x2/2 max-pool on PF, 8 channels / thread
// Scan order (0,0),(0,1),(1,0),(1,1); strict '>' so the first maximum wins, NaN wins (max_pool2d_with_indices).
// IDX = the type of the flat element index: unsigned 32-bit whenever the tensor allows it (64-bit divisions cost
// ~100 instructions each and there are three per element; with them the kernel ran at 0.6 of the copy bandwidth)
template <typename IDX>
__global__ void maxpool2_pf_kernel(const uint4* __restrict__ act, const uint4* __restrict__ gain,
                                   uint4* __restrict__ pooled, uint2* __restrict__ idx, uint4* __restrict__ gpool,
                                   int n, int h, int w, int c8) {
  const int oh = h / 2, ow = w / 2;
  const int wp1 = w + 1, owp1 = ow + 1;
  const IDX blk_f = (IDX)(h + 1) * wp1, blk_p = (IDX)(oh + 1) * owp1;
  const IDX total = (IDX)n * blk_p * c8;
  for (IDX i = blockIdx.x * (IDX)blockDim.x + threadIdx.x; i < total; i += (IDX)gridDim.x * blockDim.x) {
    const IDX prow = i / (IDX)c8;
    int cc = (int)(i - prow * c8);
    const IDX img_ = prow / blk_p;
    int img = (int)img_, rem = (int)(prow - img_ * blk_p);
    int a = rem / owp1, b = rem - a * owp1;
    uint4 outv = make_uint4(0, 0, 0, 0), outg = make_uint4(0, 0, 0, 0);
    uint2 pk = make_uint2(0, 0);
    if (a > 0 && b > 0) {
      // pooled pixel (a-1, b-1) covers fine PF rows 2a-1, 2a and columns 2b-1, 2b
      size_t base = ((size_t)img * blk_f + (size_t)(2 * a - 1) * wp1 + (2 * b - 1)) * c8 + cc;
      size_t off[4] = {base, base + c8, base + (size_t)wp1 * c8, base + (size_t)wp1 * c8 + c8};
      uint4 v[4], g[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        v[k] = act[off[k]];
        g[k] = gain ? gain[off[k]] : make_uint4(0, 0, 0, 0);
      }
      // everything below indexes registers with compile-time constants only: a run-time index into v[] / g[] (e.g.
      // v[best_k]) would move both arrays to local memory — measured: 0.6 of the copy bandwidth with that form
      const uint32_t vw[4][4] = {{v[0].x, v[0].y, v[0].z, v[0].w}, {v[1].x, v[1].y, v[1].z, v[1].w},
                                 {v[2].x, v[2].y, v[2].z, v[2].w}, {v[3].x, v[3].y, v[3].z, v[3].w}};
      const uint32_t gw[4][4] = {{g[0].x, g[0].y, g[0].z, g[0].w}, {g[1].x, g[1].y, g[1].z, g[1].w},
                                 {g[2].x, g[2].y, g[2].z, g[2].w}, {g[3].x, g[3].y, g[3].z, g[3].w}};
      uint32_t ovw[4], ogw[4], biw[2] = {0u, 0u};
#pragma unroll
      for (int wd = 0; wd < 4; ++wd) {                 // word wd holds channels 2*wd (low half) and 2*wd+1 (high half)
        uint32_t o_v = 0u, o_g = 0u;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const int sh = 16 * hf;
          float best = -INFINITY;
          uint32_t bv = 0u, bg = 0u, bk = 0u;
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t bits = (vw[k][wd] >> sh) & 0xFFFFu;
            const float f = __uint_as_float(bits << 16);
            if (f > best || f != f) { best = f; bv = bits; bg = (gw[k][wd] >> sh) & 0xFFFFu; bk = (uint32_t)k; }
          }
          o_v |= bv << sh;
          o_g |= bg << sh;
          const int e = 2 * wd + hf;
          biw[e >> 2] |= bk << (8 * (e & 3));
        }
        ovw[wd] = o_v;
        ogw[wd] = o_g;
      }
      outv = make_uint4(ovw[0], ovw[1], ovw[2], ovw[3]);
      outg = make_uint4(ogw[0], ogw[1], ogw[2], ogw[3]);
      pk.x = biw[0];
      pk.y = biw[1];
    }
    pooled[i] = outv;
    if (idx) idx[i] = pk;
    if (gpool) gpool[i] = outg;
  }
}

// ---------------------------------------------------------------- chain entry: s_top = r * rz  (fp32 -> PF bf16)
__global__ void scale_rows_kernel(const float* __restrict__ r, const uint4* __restrict__ rz,
                                  const int32_t* __restrict__ row_img, uint4* __restrict__ out, int h, int w, int c8,
                                  long long total) {
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int cc = (int)(i % c8);
    long long prow = i / c8;
    int e = (int)(prow / blk), rem = (int)(prow % blk);
    int a = rem / wp1, b = rem % wp1;
    uint4 o = make_uint4(0, 0, 0, 0);
    if (a > 0 && b > 0) {
      int img = row_img ? row_img[e] : e;
      uint4 g = rz[((size_t)img * blk + rem) * c8 + cc];
      const float4* rp = reinterpret_cast<const float4*>(r + (((size_t)e * h + (a - 1)) * w + (b - 1)) * (c8 * 8) + cc * 8);
      float4 r0 = rp[0], r1 = rp[1];
      const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
      const float rv[8] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y, r1.z, r1.w};
      uint32_t ow[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float lo = rv[2 * k] * __uint_as_float(gw[k] << 16);
        float hi = rv[2 * k + 1] * __uint_as_float(gw[k] & 0xFFFF0000u);
        __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
        ow[k] = *reinterpret_cast<uint32_t*>(&t);
      }
      o = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
    out[i] = o;
  }
}

// ---------------------------------------------------------------- PF <-> dense
__global__ void pf_to_dense_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int n, int h, int w,
                                   int c, int layout) {
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  long long total = (long long)n * h * w * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int ch, y, x, img;
    if (layout == 0) {
      ch = (int)(i % c);
      long long pix = i / c;
      x = (int)(pix % w); y = (int)((pix / w) % h); img = (int)(pix / ((long long)w * h));
    } else {
      x = (int)(i % w); y = (int)((i / w) % h);
      ch = (int)((i / ((long long)w * h)) % c); img = (int)(i / ((long long)w * h * c));
    }
    dst[i] = __bfloat162float(src[((size_t)img * blk + (size_t)(y + 1) * wp1 + (x + 1)) * c + ch]);
  }
}

__global__ void nchw_to_pf_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst, int n, int c, int h,
                                  int w, int c_pad) {
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  long long total = (long long)n * blk * c_pad;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int ch = (int)(i % c_pad);
    long long prow = i / c_pad;
    int img = (int)(prow / blk), rem = (int)(prow % blk);
    int a = rem / wp1, b = rem % wp1;
    float v = 0.f;
    if (a > 0 && b > 0 && ch < c) v = src[(((size_t)img * c + ch) * h + (a - 1)) * w + (b - 1)];
    dst[i] = __float2bfloat16(v);
  }
}

// ---------------------------------------------------------------- first layer as a tensor-core GEMM: sign-split im2col
// PF row of pixel (y,x) <- 64 bf16: [x+ over the 27 (ci,r,s) taps | x- over the 27 taps | 10 zeros], so that the
// first conv is a 1x1 "convolution" with K = 64 for lrpx_tc_conv(EPI_FWD_GAIN): rows [w | w | 0] give z = W*x and
// rows [w+ | w- | 0] give z+ = W+*x+ + W-*x- (lrp_modules.py:81-84).
__global__ void im2col3_split_kernel(const float* __restrict__ x, uint32_t* __restrict__ dst, int n, int h, int w) {
  // one thread per PF row: 27 coalesced loads (consecutive lanes = consecutive pixels), all tap arithmetic static
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  const long long total = (long long)n * blk;
  for (long long prow = blockIdx.x * (long long)blockDim.x + threadIdx.x; prow < total;
       prow += (long long)gridDim.x * blockDim.x) {
    const int img = (int)(prow / blk), rem = (int)(prow % blk);
    const int a = rem / wp1, b = rem % wp1;
    uint32_t o[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) o[j] = 0u;
    if (a > 0 && b > 0) {
      const float* xi = x + (size_t)img * 3 * h * w;
      float v[28];
      v[27] = 0.f;
#pragma unroll
      for (int k = 0; k < 27; ++k) {
        const int ci = k / 9, r = (k % 9) / 3, s = k % 3;
        const int yy = a - 1 + r - 1, xs = b - 1 + s - 1;
        v[k] = (yy >= 0 && yy < h && xs >= 0 && xs < w) ? __ldg(xi + ((size_t)ci * h + yy) * w + xs) : 0.f;
      }
      // columns 0..26 = x+, 27..53 = x-, 54..63 = 0
#pragma unroll
      for (int j = 0; j < 27; ++j) {
        const int e0 = 2 * j, e1 = 2 * j + 1;
        const float f0 = e0 < 27 ? fmaxf(v[e0], 0.f) : fminf(v[e0 - 27], 0.f);
        const float f1 = e1 < 27 ? fmaxf(v[e1], 0.f) : fminf(v[e1 - 27], 0.f);
        __nv_bfloat162 t = __floats2bfloat162_rn(f0, f1);
        o[j] = *reinterpret_cast<uint32_t*>(&t);
      }
    }
    uint32_t* d = dst + prow * 32;
#pragma unroll
    for (int q = 0; q < 4; ++q)
      asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(d + 8 * q), "r"(o[8 * q]),
                   "r"(o[8 * q + 1]), "r"(o[8 * q + 2]), "r"(o[8 * q + 3]), "r"(o[8 * q + 4]), "r"(o[8 * q + 5]),
                   "r"(o[8 * q + 6]), "r"(o[8 * q + 7])
                   : "memory");
  }
}


// ---------------------------------------------------------------- companions of the general (groups / split) modes
// A hi|lo split row of C logical channels holds 2*C bf16: [hi(0..C) | lo(0..C)], value = hi + lo (16 significant bits).
__device__ __forceinline__ void split2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
  hi = *reinterpret_cast<uint32_t*>(&h);
  __nv_bfloat162 l = __floats2bfloat162_rn(v0 - __uint_as_float(hi << 16), v1 - __uint_as_float(hi & 0xFFFF0000u));
  lo = *reinterpret_cast<uint32_t*>(&l);
}
__device__ __forceinline__ float bf_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// sign-split im2col with hi|lo rows: 128 columns [hi of the 64 | lo of the 64].  One thread per PF row like
// im2col3_split_kernel above (27 coalesced loads, all tap arithmetic static); the row leaves as eight 32-byte stores.
// (The first version — one thread per 8 columns with per-column div / mod tap arithmetic — took 0.66 ms for 64 images
// against 0.11 ms of the bf16 kernel for twice the bytes.)
__global__ void im2col3_split_x_kernel(const float* __restrict__ x, uint32_t* __restrict__ dst, int n, int h, int w) {
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  const long long total = (long long)n * blk;
  for (long long prow = blockIdx.x * (long long)blockDim.x + threadIdx.x; prow < total;
       prow += (long long)gridDim.x * blockDim.x) {
    const int img = (int)(prow / blk), rem = (int)(prow % blk);
    const int a = rem / wp1, b = rem % wp1;
    uint32_t hi[32], lo[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) hi[j] = lo[j] = 0u;
    if (a > 0 && b > 0) {
      const float* xi = x + (size_t)img * 3 * h * w;
      float v[28];
      v[27] = 0.f;
#pragma unroll
      for (int k = 0; k < 27; ++k) {
        const int ci = k / 9, r = (k % 9) / 3, ss = k % 3;
        const int yy = a - 1 + r - 1, xs = b - 1 + ss - 1;
        v[k] = (yy >= 0 && yy < h && xs >= 0 && xs < w) ? __ldg(xi + ((size_t)ci * h + yy) * w + xs) : 0.f;
      }
      // columns 0..26 = x+, 27..53 = x-, 54..63 = 0
#pragma unroll
      for (int j = 0; j < 27; ++j) {
        const int e0 = 2 * j, e1 = 2 * j + 1;
        const float f0 = e0 < 27 ? fmaxf(v[e0], 0.f) : fminf(v[e0 - 27], 0.f);
        const float f1 = e1 < 27 ? fmaxf(v[e1], 0.f) : fminf(v[e1 - 27], 0.f);
        split2(f0, f1, hi[j], lo[j]);
      }
    }
    uint32_t* d = dst + prow * 64;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(d + 8 * q), "r"(hi[8 * q]),
                   "r"(hi[8 * q + 1]), "r"(hi[8 * q + 2]), "r"(hi[8 * q + 3]), "r"(hi[8 * q + 4]), "r"(hi[8 * q + 5]),
                   "r"(hi[8 * q + 6]), "r"(hi[8 * q + 7])
                   : "memory");
      asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(d + 32 + 8 * q), "r"(lo[8 * q]),
                   "r"(lo[8 * q + 1]), "r"(lo[8 * q + 2]), "r"(lo[8 * q + 3]), "r"(lo[8 * q + 4]), "r"(lo[8 * q + 5]),
                   "r"(lo[8 * q + 6]), "r"(lo[8 * q + 7])
                   : "memory");
    }
  }
}

// 2x2/2 max-pool, 8 channels per thread, for bf16 or hi|lo rows and up to two gain tensors (bf16, or fp32 with split).
// Scan order (0,0),(0,1),(1,0),(1,1); strict '>' so the first maximum wins, NaN wins (max_pool2d_with_indices).
template <bool SPLIT>
__global__ void maxpool2_x_kernel(const uint4* __restrict__ act, const void* __restrict__ g0, const void* __restrict__ g1,
                                  uint4* __restrict__ pooled, uint2* __restrict__ idx, void* __restrict__ gp0,
                                  void* __restrict__ gp1, int n, int h, int w, int c8) {
  const int oh = h / 2, ow = w / 2;
  const int wp1 = w + 1, owp1 = ow + 1;
  const long long blk_f = (long long)(h + 1) * wp1, blk_p = (long long)(oh + 1) * owp1;
  const long long total = (long long)n * blk_p * c8;
  const int rowv = SPLIT ? 2 * c8 : c8;            // uint4 per activation row
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long prow = i / c8;
    const int cc = (int)(i - prow * c8);
    const long long img = prow / blk_p;
    const int rem = (int)(prow - img * blk_p);
    const int a = rem / owp1, b = rem - a * owp1;
    uint32_t ohi[4] = {0u, 0u, 0u, 0u}, olo[4] = {0u, 0u, 0u, 0u};
    uint32_t bidx[8];
    float og0[8], og1[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) { bidx[e] = 0u; og0[e] = 0.f; og1[e] = 0.f; }
    if (a > 0 && b > 0) {
      const long long frow0 = img * blk_f + (long long)(2 * a - 1) * wp1 + (2 * b - 1);
      const long long frow[4] = {frow0, frow0 + 1, frow0 + wp1, frow0 + wp1 + 1};
      float best[8];
      uint32_t bh[8], bl[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { best[e] = -INFINITY; bh[e] = 0u; bl[e] = 0u; }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint4 vh = act[frow[k] * rowv + cc];
        const uint4 vl = SPLIT ? act[frow[k] * rowv + c8 + cc] : make_uint4(0u, 0u, 0u, 0u);
        const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w}, lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const uint32_t hb = (hw[e >> 1] >> (16 * (e & 1))) & 0xFFFFu, lb = (lw[e >> 1] >> (16 * (e & 1))) & 0xFFFFu;
          const float f = __uint_as_float(hb << 16) + __uint_as_float(lb << 16);
          if (f > best[e] || f != f) { best[e] = f; bh[e] = hb; bl[e] = lb; bidx[e] = (uint32_t)k; }
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        ohi[e >> 1] |= bh[e] << (16 * (e & 1));
        olo[e >> 1] |= bl[e] << (16 * (e & 1));
      }
      // gains gathered at the winner (run-time row choice through the pointer, not through a register array)
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const long long fr = frow0 + (bidx[e] >> 1) * wp1 + (bidx[e] & 1);
        const size_t go = (size_t)fr * (c8 * 8) + cc * 8 + e;
        if (SPLIT) {
          if (g0) og0[e] = __ldg(reinterpret_cast<const float*>(g0) + go);
          if (g1) og1[e] = __ldg(reinterpret_cast<const float*>(g1) + go);
        } else {
          if (g0) og0[e] = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(g0)[go]);
          if (g1) og1[e] = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(g1)[go]);
        }
      }
    }
    pooled[prow * rowv + cc] = make_uint4(ohi[0], ohi[1], ohi[2], ohi[3]);
    if (SPLIT) pooled[prow * rowv + c8 + cc] = make_uint4(olo[0], olo[1], olo[2], olo[3]);
    if (idx) idx[i] = make_uint2(bidx[0] | (bidx[1] << 8) | (bidx[2] << 16) | (bidx[3] << 24),
                                 bidx[4] | (bidx[5] << 8) | (bidx[6] << 16) | (bidx[7] << 24));
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      void* gp = j ? gp1 : gp0;
      const float* og = j ? og1 : og0;
      if (!gp) continue;
      if (SPLIT) {
        float4* d = reinterpret_cast<float4*>(reinterpret_cast<float*>(gp) + (size_t)i * 8);
        d[0] = make_float4(og[0], og[1], og[2], og[3]);
        d[1] = make_float4(og[4], og[5], og[6], og[7]);
      } else {
        uint32_t wv[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          __nv_bfloat162 t = __floats2bfloat162_rn(og[2 * k], og[2 * k + 1]);
          wv[k] = *reinterpret_cast<uint32_t*>(&t);
        }
        reinterpret_cast<uint4*>(gp)[i] = make_uint4(wv[0], wv[1], wv[2], wv[3]);
      }
    }
  }
}

// chain entry of the general modes: out row = [r*rz0 | r*rz1] (groups) as bf16 or hi|lo
template <bool SPLIT>
__global__ void scale_rows_x_kernel(const float* __restrict__ r, const void* __restrict__ rz0, const void* __restrict__ rz1,
                                    const int32_t* __restrict__ row_img, uint4* __restrict__ out, int h, int w, int c8,
                                    int groups, long long total, bool clamp) {
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  const int rowv = c8 * groups * (SPLIT ? 2 : 1);
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cc = (int)(i % c8);
    const long long prow = i / c8;
    const int e = (int)(prow / blk), rem = (int)(prow % blk);
    const int a = rem / wp1, b = rem % wp1;
    const bool valid = a > 0 && b > 0;
    float rv[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) rv[k] = 0.f;
    int img = 0;
    if (valid) {
      img = row_img ? row_img[e] : e;
      const float4* rp = reinterpret_cast<const float4*>(r + (((size_t)e * h + (a - 1)) * w + (b - 1)) * (c8 * 8) + cc * 8);
      const float4 r0 = rp[0], r1 = rp[1];
      rv[0] = r0.x; rv[1] = r0.y; rv[2] = r0.z; rv[3] = r0.w; rv[4] = r1.x; rv[5] = r1.y; rv[6] = r1.z; rv[7] = r1.w;
      if (clamp)        // guided backpropagation: the last ReLU passes only the positive part (gridTDmodel.py:1684)
#pragma unroll
        for (int k = 0; k < 8; ++k) rv[k] = fmaxf(rv[k], 0.f);
    }
    for (int j = 0; j < groups; ++j) {
      const void* rz = j ? rz1 : rz0;
      float gz[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) gz[k] = 0.f;
      if (valid) {
        const size_t go = ((size_t)img * blk + rem) * (c8 * 8) + cc * 8;
        if (SPLIT) {
          const float4* gp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(rz) + go);
          const float4 g0 = gp[0], g1 = gp[1];
          gz[0] = g0.x; gz[1] = g0.y; gz[2] = g0.z; gz[3] = g0.w; gz[4] = g1.x; gz[5] = g1.y; gz[6] = g1.z; gz[7] = g1.w;
        } else {
          const uint4 g = *reinterpret_cast<const uint4*>(reinterpret_cast<const __nv_bfloat16*>(rz) + go);
          const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
          for (int k = 0; k < 4; ++k) { gz[2 * k] = bf_lo(gw[k]); gz[2 * k + 1] = bf_hi(gw[k]); }
        }
      }
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) split2(rv[2 * k] * gz[2 * k], rv[2 * k + 1] * gz[2 * k + 1], hi[k], lo[k]);
      out[prow * rowv + (size_t)j * c8 + cc] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      if (SPLIT) out[prow * rowv + (size_t)(groups + j) * c8 + cc] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
  }
}

__global__ void pf_split_to_dense_kernel(const __nv_bfloat16* __restrict__ src, float* __restrict__ dst, int n, int h,
                                         int w, int c, int layout) {
  const int wp1 = w + 1, blk = (h + 1) * wp1;
  long long total = (long long)n * h * w * c;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    int ch, y, x, img;
    if (layout == 0) {
      ch = (int)(i % c);
      long long pix = i / c;
      x = (int)(pix % w); y = (int)((pix / w) % h); img = (int)(pix / ((long long)w * h));
    } else {
      x = (int)(i % w); y = (int)((i / w) % h);
      ch = (int)((i / ((long long)w * h)) % c); img = (int)(i / ((long long)w * h * c));
    }
    const size_t o = ((size_t)img * blk + (size_t)(y + 1) * wp1 + (x + 1)) * (2 * c) + ch;
    dst[i] = __bfloat162float(src[o]) + __bfloat162float(src[o + c]);
  }
}


// fp32 rows (pitch lda) -> bf16 rows of 2K [hi | lo]: the A operand of an error-compensated GEMM (a_phys = 2K, cin = 3K)
__global__ void split2_rows_kernel(const float* __restrict__ x, int lda, uint4* __restrict__ out, long long rows, int k8) {
  const long long total = rows * k8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / k8;
    const int cg = (int)(i - r * k8);
    const float4* src = reinterpret_cast<const float4*>(x + r * lda + cg * 8);
    const float4 a = src[0], b = src[1];
    const float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
    out[r * 2 * k8 + cg] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    out[r * 2 * k8 + k8 + cg] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// ---------------------------------------------------------------- ResNet stem and strides (models/resnet.py:143-239)
// conv1 = 7x7 / stride 2 / pad 3 on the mixed-sign image: sign-split im2col at the OUTPUT resolution (ho, wo) = (h/2, w/2):
// PF row of output pixel (y,x) <- 320 bf16: [x+ over the 147 (ci,ky,kx) taps | x- over the 147 taps | 26 zeros], so that the
// layer is a 1x1 "convolution" with K = 320 for lrpx_tc_conv(FWDX) with rows [w | w | 0] (z) and [w+ | w- | 0] (z+).
__global__ void im2col7s2_split_kernel(const float* __restrict__ x, uint4* __restrict__ dst, int n, int h, int w) {
  const int ho = h / 2, wo = w / 2, wp1 = wo + 1, blk = (ho + 1) * wp1;
  const long long total = (long long)n * blk * 40;          // 40 groups of 8 columns per row
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % 40);
    const long long prow = i / 40;
    const int img = (int)(prow / blk), rem = (int)(prow % blk);
    const int a = rem / wp1, b = rem % wp1;
    uint32_t o[4] = {0u, 0u, 0u, 0u};
    if (a > 0 && b > 0) {
      const float* xi = x + (size_t)img * 3 * h * w;
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int e = cg * 8 + k;
        float f = 0.f;
        if (e < 294) {
          const int t = e < 147 ? e : e - 147;
          const int ci = t / 49, ky = (t % 49) / 7, kx = t % 7;
          const int yy = 2 * (a - 1) - 3 + ky, xs = 2 * (b - 1) - 3 + kx;
          const float xv = (yy >= 0 && yy < h && xs >= 0 && xs < w) ? __ldg(xi + ((size_t)ci * h + yy) * w + xs) : 0.f;
          f = e < 147 ? fmaxf(xv, 0.f) : fminf(xv, 0.f);
        }
        v[k] = f;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        __nv_bfloat162 t2 = __floats2bfloat162_rn(v[2 * k], v[2 * k + 1]);
        o[k] = *reinterpret_cast<uint32_t*>(&t2);
      }
    }
    dst[prow * 40 + cg] = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// the same im2col with hi|lo rows: 640 bf16 [hi of the 320 | lo of the 320], hi + lo ~ the fp32 tap (the A operand of the
// error-compensated stem, a_phys = 640 under K = 960).  hi is what im2col7s2_split_kernel writes.
__global__ void im2col7s2_split_x_kernel(const float* __restrict__ x, uint4* __restrict__ dst, int n, int h, int w) {
  const int ho = h / 2, wo = w / 2, wp1 = wo + 1, blk = (ho + 1) * wp1;
  const long long total = (long long)n * blk * 40;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int cg = (int)(i % 40);
    const long long prow = i / 40;
    const int img = (int)(prow / blk), rem = (int)(prow % blk);
    const int a = rem / wp1, b = rem % wp1;
    uint32_t hi[4] = {0u, 0u, 0u, 0u}, lo[4] = {0u, 0u, 0u, 0u};
    if (a > 0 && b > 0) {
      const float* xi = x + (size_t)img * 3 * h * w;
      float v[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int e = cg * 8 + k;
        float f = 0.f;
        if (e < 294) {
          const int t = e < 147 ? e : e - 147;
          const int ci = t / 49, ky = (t % 49) / 7, kx = t % 7;
          const int yy = 2 * (a - 1) - 3 + ky, xs = 2 * (b - 1) - 3 + kx;
          const float xv = (yy >= 0 && yy < h && xs >= 0 && xs < w) ? __ldg(xi + ((size_t)ci * h + yy) * w + xs) : 0.f;
          f = e < 147 ? fmaxf(xv, 0.f) : fminf(xv, 0.f);
        }
        v[k] = f;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) split2(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
    }
    dst[prow * 80 + cg] = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    dst[prow * 80 + 40 + cg] = make_uint4(lo[0], lo[1], lo[2], lo[3]);
  }
}

// 3x3 / stride 2 / pad 1 max-pool on PF bf16 (post-ReLU input), 8 channels per thread.  Window of output (y,x): input rows
// 2y-1..2y+1, columns 2x-1..2x+1, padding skipped (PyTorch pads with -inf); scan order (ky,kx) row-major, strict '>' so
// the first maximum wins (max_pool2d_with_indices).  idx = ky*3+kx of the winner, 255 when the maximum is 0: such a
// window passes no relevance (Z = 0: R_in = X * S = 0, lrp_modules.py:186-191).
__global__ void maxpool3s2_pf_kernel(const uint4* __restrict__ act, uint4* __restrict__ pooled, uint2* __restrict__ idx,
                                     int n, int h, int w, int c8) {
  const int oh = h / 2, ow = w / 2, wp1 = w + 1, owp1 = ow + 1;
  const long long blk_f = (long long)(h + 1) * wp1, blk_p = (long long)(oh + 1) * owp1;
  const long long total = (long long)n * blk_p * c8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long prow = i / c8;
    const int cc = (int)(i - prow * c8);
    const long long img = prow / blk_p;
    const int rem = (int)(prow - img * blk_p);
    const int a = rem / owp1, b = rem - a * owp1;
    uint32_t ov[4] = {0u, 0u, 0u, 0u};
    uint32_t bi[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) bi[e] = 255u;
    if (a > 0 && b > 0) {
      float best[8];
      uint32_t bb[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { best[e] = 0.f; bb[e] = 0u; }       // inputs are >= 0: a maximum of 0 keeps idx = 255
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int fa = 2 * (a - 1) + ky;          // PF row of input row 2y-1+ky
        if (fa < 1) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int fb = 2 * (b - 1) + kx;
          if (fb < 1) continue;
          const uint4 v = act[(img * blk_f + (long long)fa * wp1 + fb) * c8 + cc];
          const uint32_t vw[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const uint32_t bits = (vw[e >> 1] >> (16 * (e & 1))) & 0xFFFFu;
            const float f = __uint_as_float(bits << 16);
            if (f > best[e]) { best[e] = f; bb[e] = bits; bi[e] = (uint32_t)(ky * 3 + kx); }
          }
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) ov[e >> 1] |= bb[e] << (16 * (e & 1));
    }
    pooled[i] = make_uint4(ov[0], ov[1], ov[2], ov[3]);
    idx[i] = make_uint2(bi[0] | (bi[1] << 8) | (bi[2] << 16) | (bi[3] << 24), bi[4] | (bi[5] << 8) | (bi[6] << 16) | (bi[7] << 24));
  }
}

// the same pool on hi|lo rows (2*c bf16 per row): the winner is the largest hi + lo (exact in fp32), same scan order and
// 255 rule; pooled keeps the winner's hi and lo.
__global__ void maxpool3s2_x_kernel(const uint4* __restrict__ act, uint4* __restrict__ pooled, uint2* __restrict__ idx,
                                    int n, int h, int w, int c8) {
  const int oh = h / 2, ow = w / 2, wp1 = w + 1, owp1 = ow + 1;
  const long long blk_f = (long long)(h + 1) * wp1, blk_p = (long long)(oh + 1) * owp1;
  const long long total = (long long)n * blk_p * c8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long prow = i / c8;
    const int cc = (int)(i - prow * c8);
    const long long img = prow / blk_p;
    const int rem = (int)(prow - img * blk_p);
    const int a = rem / owp1, b = rem - a * owp1;
    uint32_t ohi[4] = {0u, 0u, 0u, 0u}, olo[4] = {0u, 0u, 0u, 0u};
    uint32_t bi[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) bi[e] = 255u;
    if (a > 0 && b > 0) {
      float best[8];
      uint32_t bh[8], bl[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) { best[e] = 0.f; bh[e] = 0u; bl[e] = 0u; }
#pragma unroll
      for (int ky = 0; ky < 3; ++ky) {
        const int fa = 2 * (a - 1) + ky;
        if (fa < 1) continue;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int fb = 2 * (b - 1) + kx;
          if (fb < 1) continue;
          const long long fr = (img * blk_f + (long long)fa * wp1 + fb) * 2 * c8;
          const uint4 vh = act[fr + cc], vl = act[fr + c8 + cc];
          const uint32_t hw[4] = {vh.x, vh.y, vh.z, vh.w}, lw[4] = {vl.x, vl.y, vl.z, vl.w};
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const uint32_t hb = (hw[e >> 1] >> (16 * (e & 1))) & 0xFFFFu, lb = (lw[e >> 1] >> (16 * (e & 1))) & 0xFFFFu;
            const float f = __uint_as_float(hb << 16) + __uint_as_float(lb << 16);
            if (f > best[e]) { best[e] = f; bh[e] = hb; bl[e] = lb; bi[e] = (uint32_t)(ky * 3 + kx); }
          }
        }
      }
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        ohi[e >> 1] |= bh[e] << (16 * (e & 1));
        olo[e >> 1] |= bl[e] << (16 * (e & 1));
      }
    }
    pooled[prow * 2 * c8 + cc] = make_uint4(ohi[0], ohi[1], ohi[2], ohi[3]);
    pooled[prow * 2 * c8 + c8 + cc] = make_uint4(olo[0], olo[1], olo[2], olo[3]);
    idx[i] = make_uint2(bi[0] | (bi[1] << 8) | (bi[2] << 16) | (bi[3] << 24), bi[4] | (bi[5] << 8) | (bi[6] << 16) | (bi[7] << 24));
  }
}

// Relevance through that pool (gather form, deterministic for the overlapping windows) fused with the gain of the layer
// below:  out[e][i][j][c] = gain[img][i][j][c] * sum over the (up to 4) windows (y,x) that contain (i,j) and whose winner
// is (i,j) of r[e][y][x][c].   r: per-request PF (oh, ow); gain / idx: per image; out: per-request PF (h, w).
__global__ void unpool3s2_pf_kernel(const uint4* __restrict__ r, const uint2* __restrict__ idx, const uint4* __restrict__ gain,
                                    const int32_t* __restrict__ row_img, uint4* __restrict__ out, int nq, int h, int w, int c8) {
  const int oh = h / 2, ow = w / 2, wp1 = w + 1, owp1 = ow + 1;
  const long long blk_f = (long long)(h + 1) * wp1, blk_p = (long long)(oh + 1) * owp1;
  const long long total = (long long)nq * blk_f * c8;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const long long prow = t / c8;
    const int cc = (int)(t - prow * c8);
    const long long e = prow / blk_f;
    const int rem = (int)(prow - e * blk_f);
    const int a = rem / wp1, b = rem - a * wp1;
    uint32_t ow4[4] = {0u, 0u, 0u, 0u};
    if (a > 0 && b > 0) {
      const int img = row_img ? row_img[e] : (int)e;
      const int i = a - 1, j = b - 1;
      float acc[8];
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = 0.f;
      // windows: y with 2y-1 <= i <= 2y+1  <=>  y in {i/2, (i+1)/2} (deduplicated), same for x
      const int y0 = i >> 1, y1 = (i + 1) >> 1, x0 = j >> 1, x1 = (j + 1) >> 1;
      for (int yy = y0; yy <= y1; ++yy) {
        if (yy >= oh) continue;
        const int ky = i - (2 * yy - 1);
        for (int xx = x0; xx <= x1; ++xx) {
          if (xx >= ow) continue;
          const int kx = j - (2 * xx - 1);
          const uint32_t want = (uint32_t)(ky * 3 + kx);
          const long long pr = (long long)(yy + 1) * owp1 + (xx + 1);
          const uint2 id = idx[((long long)img * blk_p + pr) * c8 + cc];
          const uint4 rv = r[(e * blk_p + pr) * c8 + cc];
          const uint32_t rw[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            const uint32_t byte = ((k < 4 ? id.x : id.y) >> (8 * (k & 3))) & 0xFFu;
            if (byte == want) acc[k] += __uint_as_float(((rw[k >> 1] >> (16 * (k & 1))) & 0xFFFFu) << 16);
          }
        }
      }
      const uint4 g = gain[((long long)img * blk_f + rem) * c8 + cc];
      const uint32_t gw[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float lo = acc[2 * k] * __uint_as_float(gw[k] << 16), hi = acc[2 * k + 1] * __uint_as_float(gw[k] & 0xFFFF0000u);
        __nv_bfloat162 t2 = __floats2bfloat162_rn(lo, hi);
        ow4[k] = *reinterpret_cast<uint32_t*>(&t2);
      }
    }
    out[t] = make_uint4(ow4[0], ow4[1], ow4[2], ow4[3]);
  }
}

// dst (n, h/2, w/2) PF <- src (n, h, w) PF at the even pixels (the input of a 1x1 / stride 2 convolution)
__global__ void subsample2_pf_kernel(const uint4* __restrict__ src, uint4* __restrict__ dst, int n, int h, int w, int c8) {
  const int oh = h / 2, ow = w / 2, wp1 = w + 1, owp1 = ow + 1;
  const long long blk_f = (long long)(h + 1) * wp1, blk_p = (long long)(oh + 1) * owp1;
  const long long total = (long long)n * blk_p * c8;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long prow = i / c8;
    const int cc = (int)(i - prow * c8);
    const long long img = prow / blk_p;
    const int rem = (int)(prow - img * blk_p);
    const int a = rem / owp1, b = rem - a * owp1;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (a > 0 && b > 0) v = src[(img * blk_f + (long long)(2 * (a - 1) + 1) * wp1 + (2 * (b - 1) + 1)) * c8 + cc];
    dst[i] = v;
  }
}

// Stem relevance, second half: the 1x1 GEMM produced P[q][tap*6 + s*3 + c] = sum_ch A[q][ch] * W(s)[ch][c][ky][kx]
// (tap = ky*7+kx, s = 0: W+, 1: W-) for every output pixel q = (y,x) of conv1; the image relevance gathers
//   heat[e][c][i][j] = x+ * sum P[(y,x)][tap][0][c] + x- * sum P[(y,x)][tap][1][c]   over 2y-3+ky = i, 2x-3+kx = j
// (lrp_modules.py:81-84, utils.py:26-30 for the stride-2 convolution).  mode: 0 fp32 (n,3,h,w), 1 channel mean, 2 fp16.
template <bool PBF16>
__global__ void stem_col2im_kernel(const void* __restrict__ Pv, int ldp, const float* __restrict__ x,
                                   const int32_t* __restrict__ row_img, void* __restrict__ out, int nq, int h, int w, int mode) {
  const int ho = h / 2, wo = w / 2, wp1 = wo + 1, blk = (ho + 1) * wp1;
  const long long total = (long long)nq * h * w;
  for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int j = (int)(t % w), i = (int)((t / w) % h);
    const long long e = t / ((long long)w * h);
    const int img = row_img ? row_img[e] : (int)e;
    float cp[3] = {0.f, 0.f, 0.f}, cn[3] = {0.f, 0.f, 0.f};
    for (int ky = (i + 3) & 1; ky < 7; ky += 2) {
      const int y = (i + 3 - ky) >> 1;
      if (y < 0 || y >= ho) continue;
      for (int kx = (j + 3) & 1; kx < 7; kx += 2) {
        const int xx = (j + 3 - kx) >> 1;
        if (xx < 0 || xx >= wo) continue;
        const size_t po = ((size_t)e * blk + (size_t)(y + 1) * wp1 + (xx + 1)) * ldp + (ky * 7 + kx) * 6;
        if (PBF16) {
          const uint32_t* pr = reinterpret_cast<const uint32_t*>(reinterpret_cast<const __nv_bfloat16*>(Pv) + po);
          const uint32_t a = pr[0], b = pr[1], c = pr[2];
          cp[0] += bf_lo(a); cp[1] += bf_hi(a); cp[2] += bf_lo(b); cn[0] += bf_hi(b); cn[1] += bf_lo(c); cn[2] += bf_hi(c);
        } else {
          const float* pr = reinterpret_cast<const float*>(Pv) + po;
          const float2 p0 = *reinterpret_cast<const float2*>(pr), p1 = *reinterpret_cast<const float2*>(pr + 2),
                       p2 = *reinterpret_cast<const float2*>(pr + 4);
          cp[0] += p0.x; cp[1] += p0.y; cp[2] += p1.x; cn[0] += p1.y; cn[1] += p2.x; cn[2] += p2.y;
        }
      }
    }
    const size_t hw = (size_t)h * w, pix = (size_t)i * w + j;
    float res[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float xv = __ldg(x + ((size_t)img * 3 + c) * hw + pix);
      res[c] = fmaxf(xv, 0.f) * cp[c] + fminf(xv, 0.f) * cn[c];
    }
    if (mode == 1) {
      reinterpret_cast<float*>(out)[(size_t)e * hw + pix] = ((res[0] + res[1]) + res[2]) / 3.f;
    } else if (mode == 2) {
#pragma unroll
      for (int c = 0; c < 3; ++c) reinterpret_cast<__half*>(out)[((size_t)e * 3 + c) * hw + pix] = __float2half_rn(res[c]);
    } else {
#pragma unroll
      for (int c = 0; c < 3; ++c) reinterpret_cast<float*>(out)[((size_t)e * 3 + c) * hw + pix] = res[c];
    }
  }
}

}  // namespace lrpx

using namespace lrpx;

extern "C" {

size_t lrpx_gemm_x3_workspace_bytes(int m, int k) {
  if (m <= 0 || k <= 0) return 0;
  return (size_t)m * 2 * k * sizeof(__nv_bfloat16);
}

int lrpx_gemm_x3_f32(const float* a, int lda, const void* w3, int n_pad, const float* bias, float* out, int ldo, int m, int n,
                     int k, void* workspace, size_t workspace_bytes, void* stream) {
  LRPX_CHECK_ARG(a && w3 && out && m > 0 && n > 0 && k > 0, "bad argument");
  LRPX_CHECK_ARG(k % 64 == 0 && lda >= k && lda % 4 == 0 && n % 4 == 0 && ldo >= n && ldo % 4 == 0, "k % 64, n % 4, pitches % 4");
  LRPX_CHECK_ARG(n_pad >= n && n_pad % 32 == 0 && (n_pad <= 256 || n_pad % 256 == 0), "n_pad: multiple of 32 (<= 256) or of 256");
  LRPX_CHECK_ARG(workspace && workspace_bytes >= lrpx_gemm_x3_workspace_bytes(m, k), "workspace too small");
  LRPX_CHECK_ARG((reinterpret_cast<uintptr_t>(a) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0, "a / out must be 16-byte aligned");
  split2_rows_kernel<<<grid_for((long long)m * (k / 8)), 256, 0, as_stream(stream)>>>(a, lda, (uint4*)workspace, m, k / 8);
  LRPX_CHECK_LAUNCH();
  lrpx_tc_conv_args g{};
  g.n_img = 1; g.h = 0; g.w = m - 1; g.cin = 3 * k; g.a_phys = 2 * k; g.ncol = n_pad; g.ksize = 1;
  g.epilogue = LRPX_TC_EPI_STORE_F32;
  g.a = workspace; g.wt = w3; g.out = out; g.bias = bias; g.out_pitch = ldo; g.n_valid = n;
  return lrpx_tc_conv(&g, stream);
}

int lrpx_tc_im2col7s2_split_bf16(const float* x, void* dst, int n, int h, int w, void* stream) {
  LRPX_CHECK_ARG(x && dst && n > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0, "bad argument (h, w even)");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * 40;
  im2col7s2_split_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(x, (uint4*)dst, n, h, w);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_maxpool3s2_bf16(const void* act, void* pooled, uint8_t* idx, int n, int h, int w, int c, void* stream) {
  LRPX_CHECK_ARG(act && pooled && idx && n > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && c % 8 == 0, "bad argument");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * (c / 8);
  maxpool3s2_pf_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>((const uint4*)act, (uint4*)pooled, (uint2*)idx, n, h, w, c / 8);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_unpool3s2_bf16(const void* r, const uint8_t* idx, const void* gain, const int32_t* row_img, void* out, int n_expl,
                           int h, int w, int c, void* stream) {
  LRPX_CHECK_ARG(r && idx && gain && out && n_expl > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && c % 8 == 0, "bad argument");
  long long total = (long long)n_expl * (h + 1) * (w + 1) * (c / 8);
  unpool3s2_pf_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>((const uint4*)r, (const uint2*)idx, (const uint4*)gain,
                                                                     row_img, (uint4*)out, n_expl, h, w, c / 8);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_subsample2_bf16(const void* src, void* dst, int n, int h, int w, int c, void* stream) {
  LRPX_CHECK_ARG(src && dst && n > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && c % 8 == 0, "bad argument");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * (c / 8);
  subsample2_pf_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>((const uint4*)src, (uint4*)dst, n, h, w, c / 8);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_im2col7s2_split_x(const float* x, void* dst, int n, int h, int w, int split, void* stream) {
  if (!split) return lrpx_tc_im2col7s2_split_bf16(x, dst, n, h, w, stream);
  LRPX_CHECK_ARG(x && dst && n > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0, "bad argument (h, w even)");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * 40;
  im2col7s2_split_x_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(x, (uint4*)dst, n, h, w);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_maxpool3s2_x(const void* act, void* pooled, uint8_t* idx, int n, int h, int w, int c, int split, void* stream) {
  if (!split) return lrpx_tc_maxpool3s2_bf16(act, pooled, idx, n, h, w, c, stream);
  LRPX_CHECK_ARG(act && pooled && idx && n > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && c % 8 == 0, "bad argument");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * (c / 8);
  maxpool3s2_x_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>((const uint4*)act, (uint4*)pooled, (uint2*)idx, n, h, w, c / 8);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_stem_col2im_f32(const float* P, int ldp, const float* x, const int32_t* row_img, void* out, int n_expl, int h,
                            int w, int mode, void* stream) {
  LRPX_CHECK_ARG(P && x && out && n_expl > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && ldp >= 294 && ldp % 2 == 0 &&
                     mode >= 0 && mode <= 2, "bad argument");
  long long total = (long long)n_expl * h * w;
  stem_col2im_kernel<false><<<grid_for(total), 256, 0, as_stream(stream)>>>(P, ldp, x, row_img, out, n_expl, h, w, mode);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_stem_col2im_bf16(const void* P, int ldp, const float* x, const int32_t* row_img, void* out, int n_expl, int h,
                             int w, int mode, void* stream) {
  LRPX_CHECK_ARG(P && x && out && n_expl > 0 && h > 0 && w > 0 && h % 2 == 0 && w % 2 == 0 && ldp >= 294 && ldp % 2 == 0 &&
                     mode >= 0 && mode <= 2, "bad argument");
  long long total = (long long)n_expl * h * w;
  stem_col2im_kernel<true><<<grid_for(total), 256, 0, as_stream(stream)>>>(P, ldp, x, row_img, out, n_expl, h, w, mode);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_im2col3_split_x(const float* x, void* dst, int n, int h, int w, int split, void* stream) {
  if (!split) return lrpx_tc_im2col3_split_bf16(x, dst, n, h, w, stream);
  LRPX_CHECK_ARG(x && dst && n > 0 && h > 0 && w > 0, "bad argument");
  long long total = (long long)n * (h + 1) * (w + 1);
  im2col3_split_x_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(x, (uint32_t*)dst, n, h, w);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_maxpool2_x(const void* act, const void* gain0_fine, const void* gain1_fine, void* pooled, uint8_t* idx,
                       void* gain0_pooled, void* gain1_pooled, int n, int h, int w, int c, int split, void* stream) {
  LRPX_CHECK_ARG(act && pooled && n > 0 && h > 0 && w > 0 && c > 0 && (h % 2) == 0 && (w % 2) == 0 && (c % 8) == 0,
                 "bad argument (h, w even and c % 8 == 0 required)");
  LRPX_CHECK_ARG((gain0_fine == nullptr) == (gain0_pooled == nullptr) && (gain1_fine == nullptr) == (gain1_pooled == nullptr),
                 "fine and pooled gains go together");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * (c / 8);
  if (split)
    maxpool2_x_kernel<true><<<grid_for(total), 256, 0, as_stream(stream)>>>((const uint4*)act, gain0_fine, gain1_fine,
        (uint4*)pooled, (uint2*)idx, gain0_pooled, gain1_pooled, n, h, w, c / 8);
  else
    maxpool2_x_kernel<false><<<grid_for(total), 256, 0, as_stream(stream)>>>((const uint4*)act, gain0_fine, gain1_fine,
        (uint4*)pooled, (uint2*)idx, gain0_pooled, gain1_pooled, n, h, w, c / 8);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_scale_rows_x(const float* r, const void* rz0, const void* rz1, const int32_t* row_img, void* out,
                         int n_expl, int h, int w, int c, int groups, int split, void* stream) {
  LRPX_CHECK_ARG(r && rz0 && out && n_expl > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0, "bad argument");
  LRPX_CHECK_ARG(groups == 1 || (groups == 2 && rz1), "groups must be 1, or 2 with rz1");
  long long total = (long long)n_expl * (h + 1) * (w + 1) * (c / 8);
  const bool clamp = (split & 2) != 0;
  if (split & 1)
    scale_rows_x_kernel<true><<<grid_for(total), 256, 0, as_stream(stream)>>>(r, rz0, rz1, row_img, (uint4*)out, h, w,
                                                                             c / 8, groups, total, clamp);
  else
    scale_rows_x_kernel<false><<<grid_for(total), 256, 0, as_stream(stream)>>>(r, rz0, rz1, row_img, (uint4*)out, h, w,
                                                                              c / 8, groups, total, clamp);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_pf_split_to_dense_f32(const void* src, float* dst, int n, int h, int w, int c, int layout, void* stream) {
  LRPX_CHECK_ARG(src && dst && n > 0 && h > 0 && w > 0 && c > 0 && (layout == 0 || layout == 1), "bad argument");
  long long total = (long long)n * h * w * c;
  pf_split_to_dense_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>((const __nv_bfloat16*)src, dst, n, h, w, c, layout);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_im2col3_split_bf16(const float* x, void* dst, int n, int h, int w, void* stream) {
  LRPX_CHECK_ARG(x && dst && n > 0 && h > 0 && w > 0, "bad argument");
  long long total = (long long)n * (h + 1) * (w + 1);
  im2col3_split_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(x, (uint32_t*)dst, n, h, w);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_weight_prep_bf16(const float* w, void* wt, int cout, int cin, int kh, int kw, int mode, int rows_pad,
                          int chan_pad, void* stream) {
  LRPX_CHECK_ARG(w && wt && cout > 0 && cin > 0 && kh > 0 && kw > 0 && mode >= 0 && mode <= 3, "bad argument");
  int rows = mode >= 2 ? cin : cout, chans = mode >= 2 ? cout : cin;
  LRPX_CHECK_ARG(rows_pad >= rows && chan_pad >= chans, "padding smaller than the source");
  long long total = (long long)rows_pad * kh * kw * chan_pad;
  weight_prep_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(w, (__nv_bfloat16*)wt, cout, cin, kh, kw, mode,
                                                                    rows_pad, chan_pad);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_first_fwd(const float* x, const float* w, const float* bias, void* act, void* gain, int n, int h, int wd,
                      int cout, void* stream) {
  LRPX_CHECK_ARG(x && w && act && gain && n > 0 && h > 0 && wd > 0, "bad argument");
  LRPX_CHECK_ARG(cout == 64 || cout == 32 || cout == 16 || cout == 8, "cout must be 8, 16, 32 or 64");
  long long total = ((long long)n * (h + 1) * (wd + 1) + FF_PX - 1) / FF_PX * (cout / 8);
  size_t smem = (size_t)(3 * 27 * cout + cout) * sizeof(float);
  cudaStream_t st = as_stream(stream);
  int grid = grid_for(total);
  switch (cout) {
    case 64: first_fwd_kernel<8><<<grid, 256, smem, st>>>(x, w, bias, (uint4*)act, (uint4*)gain, n, h, wd); break;
    case 32: first_fwd_kernel<4><<<grid, 256, smem, st>>>(x, w, bias, (uint4*)act, (uint4*)gain, n, h, wd); break;
    case 16: first_fwd_kernel<2><<<grid, 256, smem, st>>>(x, w, bias, (uint4*)act, (uint4*)gain, n, h, wd); break;
    default: first_fwd_kernel<1><<<grid, 256, smem, st>>>(x, w, bias, (uint4*)act, (uint4*)gain, n, h, wd); break;
  }
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_maxpool2_bf16(const void* act, const void* gain_fine, void* pooled, uint8_t* idx, void* gain_pooled, int n,
                          int h, int w, int c, void* stream) {
  LRPX_CHECK_ARG(act && pooled && n > 0 && h > 0 && w > 0 && c > 0 && (h % 2) == 0 && (w % 2) == 0 && (c % 8) == 0,
                 "bad argument (h, w even and c % 8 == 0 required)");
  LRPX_CHECK_ARG((gain_fine == nullptr) == (gain_pooled == nullptr), "gain_fine and gain_pooled go together");
  long long total = (long long)n * (h / 2 + 1) * (w / 2 + 1) * (c / 8);
  // 32-bit indices when both the pooled element count and the fine uint4 offsets fit
  const long long fine = (long long)n * (h + 1) * (w + 1) * (c / 8);
  if (fine + 2LL * 148 * 64 * 256 < 0xFFFFFFFFLL)
    maxpool2_pf_kernel<uint32_t><<<grid_for(total), 256, 0, as_stream(stream)>>>(
        (const uint4*)act, (const uint4*)gain_fine, (uint4*)pooled, (uint2*)idx, (uint4*)gain_pooled, n, h, w, c / 8);
  else
    maxpool2_pf_kernel<long long><<<grid_for(total), 256, 0, as_stream(stream)>>>(
        (const uint4*)act, (const uint4*)gain_fine, (uint4*)pooled, (uint2*)idx, (uint4*)gain_pooled, n, h, w, c / 8);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_scale_rows(const float* r, const void* rz, const int32_t* row_img, void* out, int n_expl, int h, int w,
                       int c, void* stream) {
  LRPX_CHECK_ARG(r && rz && out && n_expl > 0 && h > 0 && w > 0 && c > 0 && c % 8 == 0, "bad argument");
  long long total = (long long)n_expl * (h + 1) * (w + 1) * (c / 8);
  scale_rows_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(r, (const uint4*)rz, row_img, (uint4*)out, h, w,
                                                                   c / 8, total);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_pf_to_dense_f32(const void* src, float* dst, int n, int h, int w, int c, int layout, void* stream) {
  LRPX_CHECK_ARG(src && dst && n > 0 && h > 0 && w > 0 && c > 0 && (layout == 0 || layout == 1), "bad argument");
  long long total = (long long)n * h * w * c;
  pf_to_dense_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>((const __nv_bfloat16*)src, dst, n, h, w, c, layout);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

int lrpx_tc_nchw_to_pf_bf16(const float* src, void* dst, int n, int c, int h, int w, int c_pad, void* stream) {
  LRPX_CHECK_ARG(src && dst && n > 0 && c > 0 && h > 0 && w > 0 && c_pad >= c, "bad argument");
  long long total = (long long)n * (h + 1) * (w + 1) * c_pad;
  nchw_to_pf_kernel<<<grid_for(total), 256, 0, as_stream(stream)>>>(src, (__nv_bfloat16*)dst, n, c, h, w, c_pad);
  LRPX_CHECK_LAUNCH();
  return LRPX_OK;
}

}  // extern "C"
