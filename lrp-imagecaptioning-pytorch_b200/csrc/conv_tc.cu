// Tensor-core relevance / forward convolution for sm_100a: tcgen05.mma (bf16 x bf16 -> fp32 in TMEM),
// operands staged by TMA (cp.async.bulk.tensor, SWIZZLE_128B), persistent warp-specialised CTAs.
//
// Reference arithmetic being replaced (per 3x3/stride-1/pad-1 conv layer, alpha=1 beta=0):
//   LRPtools/lrp_modules.py:81-84   z+ = conv(a+, W+) + conv(a-, W-)
//   LRPtools/utils.py:16-18,26-30   s = R / (z+ + 1e-7*[z+ == 0]);  c = d z+/d a (s);  R_in = a (.) c
//   LRPtools/lrp_modules.py:186-191 max-pool winner-take-all
//
// Data layout ("PF", padded-flat NHWC bf16).  An image of h x w pixels and C channels is a block of
// (h+1)*(w+1) pixel rows of C bf16 each; block row 0 and block column 0 are zero padding, pixel (y,x)
// lives at block offset (y+1)*(w+1) + (x+1).  The right/bottom halo of an image is the left/top padding of
// what follows, so for a flat pixel index p the 3x3 neighbour (dy,dx) is simply row p + dy*(w+1) + dx and
// a 3x3 convolution is 9 accumulated GEMMs over row-shifted views of ONE 2-D tensor (rows x channels):
// no im2col, every TMA box is a plain 2-D tile, out-of-range rows are zero-filled by TMA.
//
// GEMM:  acc[p][n] = sum_{tap, c} A[p + off(tap)][c] * Wt[n][tap*cin + c]      (both operands K-major)
//   tile 128 or 256 (pixels) x BN (<=256) per CTA iteration, K step 64 channels (one 128-byte swizzle row),
//   tcgen05.mma.cta_group::1.kind::f16  M=128, N=BN, K=16 (4 per K step), accumulators double-buffered in
//   TMEM (2 x 256 columns) so the epilogue of tile i overlaps the main loop of tile i+1.
// Two kernels:
//   tc_conv_kernel       one TMA tile per filter tap (1x1 convolutions / plain GEMMs: first-layer forward, decoder GEMMs)
//   tc_conv_slab_kernel  3x3: the A rows of all taps fetched once per channel block ("slab"), taps = row-shifted
//                        descriptor views; B streamed (TMA-multicast to a CTA pair) or resident; two lockstep MMA issuers
// Warp roles (20 warps): 0 = A producer, 1 = TMEM allocator + MMA issuer, 2..17 = epilogue (TMEM lane quarter =
//   warp_idx % 4, four warps per quarter share the tile's 32x32 units), 18 = B producer, 19 = second MMA issuer.
// DESIGN.md section 4.1 has the measurements behind each of these choices.
#include "lrpx_common.cuh"
#include <cuda.h>
#include <cuda_fp16.h>
#include <mutex>
#include <stdlib.h>

namespace lrpx {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;             // channels per K step (128 bytes of bf16)
constexpr int TC_MAX_STAGES = 12;
constexpr int TC_EPI_WARPS = 16;           // four warps per TMEM lane quarter, sharing the tile's 32x32 units round-robin
// warps: 0 A/TMA producer, 1 MMA, 2..17 epilogue, 18 B producer, 19 second MMA issuer (slab kernel)
constexpr int TC_THREADS = 32 * (TC_EPI_WARPS + 4);
constexpr int TC_BPROD_WARP = 2 + TC_EPI_WARPS;
constexpr int TC_MMA2_WARP = TC_BPROD_WARP + 1;
constexpr int TC_SMEM_BYTES = 220 * 1024;
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;   // 16 KiB

struct TcParams {
  int m_total;       // rows of A (n_img * blk)
  int blk;           // (h+1)*(w+1)
  int h, w;          // unpadded spatial size of A's images
  int wp1;           // w + 1
  uint32_t blk_mul, wp1_mul;   // fast_div multipliers / shifts for blk and wp1
  int blk_sh, wp1_sh;
  uint32_t nnt_mul;  // fast_div multiplier / shift for num_n_tiles (tile_coords)
  int nnt_sh;
  int cin;           // channels of A
  int ncol;          // GEMM N (rows of Wt)
  int bn;            // N tile
  int half;          // FWD_GAIN: output channels per tile (= bn/2)
  int taps;          // 1 or 9
  int kc_per_tap;    // cin / 64
  int num_m_tiles, num_n_tiles;
  int stages;
  // ---- slab mode (3x3 only): the A rows of all 9 taps of a tile are fetched once per channel block
  int slab_mode;     // 0 = off (one A tile per tap), 1 = one contiguous slab, 3 = one slab per filter row
  int mh;            // M halves per CTA tile (1 -> 128 rows, 2 -> 256 rows sharing every B tile)
  int slab_rows;     // rows per slab
  int box0_rows, box1_rows;   // TMA boxes that make up a slab (box1_rows == 0: single box)
  int a_stage_bytes; // bytes of one A stage (= one slab), multiple of 1024
  int n_issuers;     // MMA issuer warps in use: 2 (one per M half) when mh == 2, else 1
  int fold;          // EPI_INPUT3: the three filter columns are folded into N (see epi_input3); 0 otherwise
  int half_rows;     // row distance between the M halves of a tile (128; 126 with fold: the halves overlap by two rows)
  int tile_out_rows; // output rows per tile (mh*128; 252 with fold)
  int tile_stride;   // row distance between consecutive M tiles (= tile_out_rows; = w + 1 in walk mode)
  int walk;          // row walk (slab mode 3, resident B, one channel block): a CTA takes a contiguous run of tiles ONE IMAGE
                     // ROW apart, so two of a tile's three slabs are the previous tile's — see tc_conv_slab_kernel
  int tiles_per_cta; // walk: length of a CTA's run
  int a_group;       // slab mode 3: slabs per ring stage. 1 = one barrier round trip per filter row's slab; 3 = the three slabs
                     // of a tile share ONE stage (one wait + one commit per tile for the issuers, one wait for the producer)
  int nbuf_log2;     // accumulator ring of the slab kernel: 1 = two buffers of 256 TMEM columns, 2 = four of 128
  int sleep_ns;      // back-off of the producers' and the epilogue warps' barrier waits (mbar_wait_ns)
  int cluster;      // 2: CTA pairs (thread-block clusters) share every streamed B tile through TMA multicast; else 1
  int tiles_sched;   // tiles the persistent loop walks (cluster mode pads the M tiles to an even count)
  int store_off;     // EPI_MUL: byte offset (from the aligned smem base) of the TMA-store staging area, 0 = plain stores
  int a_stages, b_stages;
  int b_resident;    // all B tiles of the layer stay in shared memory for the lifetime of the CTA
  int debug_flags;   // env LRPX_TC_DEBUG: bit 0 = epilogue skips its global loads/stores (timing experiments only)
  int out_c;         // channel pitch of out / gain (elements per pixel row)
  int gain_mode;     // FWD_GAIN: 0 -> act/safe(z+), 1 -> 1/safe(z+)
  // ---- general modes (MULX / MULX_UNPOOL / FWDX)
  int a_wrap;        // physical 64-channel blocks per A row; K block kc >= a_wrap reads block kc - a_wrap (0 = no wrap)
  int groups;        // MULX*: gain groups (1 | 2)
  int split;         // 0: bf16 rows, bf16 gains; 1: hi|lo split rows, fp32 gains
  int n_acc;         // FWDX: accumulators per output channel (W [, W+ [, W-]])
  int rule;          // 0 alpha-beta, 1 epsilon, 2 gradient (gain = the ReLU's derivative), 3 guided backpropagation (as 2,
                     // and MULX passes only the positive part of the accumulator); INPUT3 with rule >= 2 returns W^T g as is
  int zbias;         // FWDX: bias enters the divisor
  int cout;          // FWDX: output channels (row pitch of the gains; act pitch = cout * (1 + split))
  float alpha, beta;
  const void* gain2;
  void* out3;
  // ---- residual-network extensions (MULX: fork sum; FWDX: folded BatchNorm, residual Add, strided store)
  const void* add;   // MULX: per-request addend rows (bf16, pitch add_pitch): out_j = acc*gain_j + add*gainB_j
  int add_pitch;
  const void* gain3; // MULX: gainB of group 0
  const void* gain4; // MULX: gainB of group 1
  const float* bn_w; // FWDX: folded BatchNorm scale / shift per output channel (nullptr: plain bias)
  const float* bn_b;
  const void* idn;   // FWDX: residual identity branch (bf16 PF, cout channels; hi|lo rows when split): Add rule ratios
  const void* hd;    // FWDX: per-element factor of the identity-branch gain (bf16 PF, fp32 when split) or nullptr
  void* out4;        // FWDX: act * gain0
  void* out5;        // FWDX: act * (identity-branch gain)
  int fwd_flags;     // FWDX: bit 0 = no ReLU, bit 1 = store only the even pixels into a half-resolution PF tensor
  int n_valid;       // STORE_F32: columns that exist in `out` (<= ncol)
  int mulx_simple;   // MULX / MULX_UNPOOL: one gain group, no addend, no second output: the _S instantiations
  int fwd_simple;    // FWDX: plain conv + bias + ReLU with one gain group (no BatchNorm fold, residual Add, strided store,
                     // extra outputs or neg-net accumulator): the short epilogue epi_fwdx_simple
  int pair;          // CTA pairs issue ONE tcgen05.mma.cta_group::2 (M = 256 = 128 rows of each CTA, each CTA holding bn/2
                     // rows of every B tile in its own shared memory): halves the B operand reads per SM
  const float* bias;
  const __nv_bfloat16* gain;
  const int32_t* row_img;
  const uint8_t* pool_idx;
  const float* x;
  const float* x1;
  void* out;
  void* out2;
  const float* cam_rows;   // INPUT3, guided rule: Guided Grad-CAM's map expanded along y (n_img, h, cam_w), or nullptr
  const float* cam_kw;     // (w, cam_w): its expansion along x
  int cam_w;
};

// ------------------------------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// Bounded wait: a broken pipeline traps (the launch fails with an error) instead of hanging the GPU.
// SLEEP_NS > 0: back off with nanosleep between polls.  Measured (ncu source view of a 512-channel layer): the 16
// epilogue warps polling their "accumulator ready" barrier executed 57 M loop trips per launch, ~1.1 instructions per
// cycle per SM of pure polling on the four schedulers the MMA issuers and TMA producers also issue from.  Waiters whose
// wake-up latency does not matter (epilogue: a tile takes ~10 us; producers: a ring stage ahead) therefore sleep;
// the MMA issuers poll without sleeping.
template <int SLEEP_NS>
__device__ __forceinline__ void mbar_wait_t(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  if (ok) return;
  long long t0 = clock64();
  for (uint32_t it = 1;; ++it) {
    if (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    if ((it & 1023) == 0 && clock64() - t0 > 4000000000LL) {
      printf("lrpx tc_conv: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) { mbar_wait_t<0>(bar, parity); }
__device__ __forceinline__ void mbar_wait_relaxed(uint32_t bar, uint32_t parity) { mbar_wait_t<200>(bar, parity); }
// the same with the back-off as a launch parameter (TcParams::sleep_ns; 0 = poll): how long a waiter may oversleep depends
// on how long a tile of the layer takes
__device__ __forceinline__ void mbar_wait_ns(uint32_t bar, uint32_t parity, uint32_t ns) {
  uint32_t ok = 0;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  if (ok) return;
  long long t0 = clock64();
  for (uint32_t it = 1;; ++it) {
    if (ns) __nanosleep(ns);
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    if (ok) return;
    if ((it & 1023) == 0 && clock64() - t0 > 4000000000LL) {
      printf("lrpx tc_conv: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// smem -> global tile store (bulk async group); the box is clipped at the tensor's bounds
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src), "r"(c0),
               "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// multicast tile load: the box lands at the same shared-memory offset in every CTA of `mask` and signals the mbarrier
// at the same offset in each of them
__device__ __forceinline__ void tma_load_2d_mc(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1,
                                               uint16_t mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], "
      "[%2], %5;" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1), "h"(mask)
      : "memory");
}
__device__ __forceinline__ void tc_commit_mc(uint32_t bar, uint16_t mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"(mask)
               : "memory");
}
// ---- 2-SM (cta_group::2) forms
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// TMA tile load into THIS CTA's shared memory that signals the mbarrier `bar` (a shared::cluster address: the leader's)
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tc_commit_2sm(uint32_t bar) {      // arrives on `bar` at the same offset in both CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
               "h"((uint16_t)3)
               : "memory");
}
__device__ __forceinline__ void tc_mma_f16_2sm(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_2d(const CUtensorMap* map, int c0, int c1) {
  asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];" ::"l"(map), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void* gptr, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gptr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// elect.sync as a C++ predicate.  ptxas recognises `if (elect_one()) { ... }` as a single-thread region whose
// values are warp-uniform: descriptors then live in uniform registers and are advanced with UIADD3, and a
// tcgen05.mma / UTMALDG costs ~3 SASS instructions.  (Measured alternatives on B200: an `if (lane == 0)` region wraps
// every UTCHMMA in an ELECT/branch loop, ~200 cycles per MMA; elect.sync predicates inside the asm statement cost
// VOTEU + 6 R2UR.BROADCAST per MMA, ~50 cycles per MMA plus ~500 per ring stage.)
__device__ __forceinline__ uint32_t elect_one() {
  uint32_t pred = 0, laneid = 0;
  asm volatile(
      "{\n\t.reg .b32 %%rx;\n\t.reg .pred %%px;\n\t"
      "elect.sync %%rx|%%px, %2;\n\t"
      "@%%px mov.s32 %1, 1;\n\t"
      "mov.s32 %0, %%rx;\n\t}"
      : "+r"(laneid), "+r"(pred)
      : "r"(0xFFFFFFFFu));
  return pred;
}
// K-major, SWIZZLE_128B shared-memory matrix descriptor: rows of 128 bytes, 8-row groups 1024 bytes apart.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address
  d |= (uint64_t)1 << 16;                          // leading-dimension byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride-dimension byte offset
  d |= (uint64_t)1 << 46;                          // descriptor version (sm_100)
  d |= (uint64_t)2 << 61;                          // SWIZZLE_128B
  return d;
}
// A row-shifted view into a slab (start address only 128-byte aligned) uses the SAME descriptor with the shifted
// start address and base offset 0: measured on B200, the 128B swizzle is a function of the absolute shared-memory
// address bits, so TMA's layout and the MMA's view agree; filling the "matrix base offset" field ((addr >> 7) & 7)
// instead produces wrong products.
// Split form for the MMA issue loops (one thread issues every MMA, so its instruction count per MMA bounds the
// tensor pipe for small N): the high word is constant, the low word is (addr >> 4) | LBO and is advanced by adds.
constexpr uint32_t TC_DESC_HI = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc_pack(uint32_t lo) { return ((uint64_t)TC_DESC_HI << 32) | (uint64_t)lo; }
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, M=128, N=bn
__device__ __forceinline__ uint32_t make_idesc(int bn, int m = TC_BM) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

#define TMEM_LD_X32(taddr, v)                                                                                   \
  asm volatile(                                                                                                 \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "                                                                 \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, "   \
      "%22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                                               \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),         \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),   \
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), \
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])  \
      : "r"(taddr)                                                                                              \
      : "memory")
#define TMEM_LD_X16(taddr, v)                                                                                   \
  asm volatile(                                                                                                 \
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "                                                                 \
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"                          \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),         \
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])    \
      : "r"(taddr)                                                                                              \
      : "memory")
#define TMEM_LD_X8(taddr, v)                                                                                    \
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"                  \
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])  \
               : "r"(taddr)                                                                                      \
               : "memory")
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
// 256-bit global accesses (sm_100): one thread moves 32 contiguous bytes per instruction.  The epilogues are
// row-per-thread (rows are >= 128 bytes apart), so every lane touches its own sector(s): wavefronts = bytes / 32.
struct U8 { uint32_t w[8]; };
__device__ __forceinline__ U8 ldg_nc_v8(const void* p) {
  U8 r;
  asm volatile("ld.global.nc.L1::no_allocate.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r.w[0]), "=r"(r.w[1]), "=r"(r.w[2]), "=r"(r.w[3]), "=r"(r.w[4]), "=r"(r.w[5]), "=r"(r.w[6]), "=r"(r.w[7])
               : "l"(p));
  return r;
}
__device__ __forceinline__ void stg_v8(void* p, const uint32_t (&w)[8]) {
  asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(w[0]), "r"(w[1]), "r"(w[2]), "r"(w[3]),
               "r"(w[4]), "r"(w[5]), "r"(w[6]), "r"(w[7])
               : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 t = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ float bf16_lo(uint32_t u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t u) { return __uint_as_float(u & 0xFFFF0000u); }

// ------------------------------------------------------------------------------------------ epilogues
// One thread owns one accumulator row (= one PF pixel).  The work of a tile is cut into UNITS of 32 rows (one TMEM
// lane quarter of one M half) x 32 columns; the four epilogue warps of a lane quarter take the units round-robin.
// (Measured on the 64-channel 224^2 layer with 8 warps and a row's whole column range per thread: the epilogue warps
// were busy 100 % of the time at ~8 cycles per instruction and ~450 instructions per 32x64 block — the epilogue, not
// the tensor pipe, set the tile time.  Hence 16 warps for latency hiding and the lean index arithmetic below.)
struct RowInfo {
  int row;       // flat PF row
  int e;         // image / explanation block
  int rem;       // offset inside the block
  int a, b;      // PF row / column inside the block (0 = padding)
  bool in_range; // row < m_total
  bool valid;    // a real pixel
};

// n / d for n < 2^31 with the host-prepared multiplier m = ceil(2^sh / d), sh = 31 + ceil(log2 d)
__device__ __forceinline__ int fast_div(int n, uint32_t m, int sh) {
  return (int)(((uint64_t)(uint32_t)n * m) >> sh);
}

__device__ __forceinline__ RowInfo row_info(const TcParams& p, int row) {
  RowInfo r;
  r.row = row;
  r.in_range = row >= 0 && row < p.m_total;
  int rr = r.in_range ? row : 0;
  r.e = fast_div(rr, p.blk_mul, p.blk_sh);
  r.rem = rr - r.e * p.blk;
  r.a = fast_div(r.rem, p.wp1_mul, p.wp1_sh);
  r.b = r.rem - r.a * p.wp1;
  r.valid = r.in_range && r.a > 0 && r.b > 0;
  return r;
}

__device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

__device__ __forceinline__ void stg_zero32(void* p) {
  const uint32_t z[8] = {0u, 0u, 0u, 0u, 0u, 0u, 0u, 0u};
  stg_v8(p, z);
}

// out[row][col..col+32) = bf16(acc * gain[img][rem][col..]);  g = the 64 bytes of gain, loaded by the caller BEFORE it
// waits on the accumulator so that the global-load latency overlaps the TMEM read
__device__ __forceinline__ void epi_mul(const TcParams& p, const RowInfo& r, int col, const uint32_t (&v)[32],
                                        const U8 (&g)[2]) {
  if (!r.in_range || (p.debug_flags & 64)) return;      // 64: timing experiment without the stores
  __nv_bfloat16* out = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)r.row * p.out_c + col;
  if (!r.valid) {          // padding rows of the PF layout stay exactly zero
    stg_zero32(out);
    stg_zero32(out + 16);
    return;
  }
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    uint32_t ow[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float a0 = __uint_as_float(v[16 * q + 2 * k]) * bf16_lo(g[q].w[k]);
      float a1 = __uint_as_float(v[16 * q + 2 * k + 1]) * bf16_hi(g[q].w[k]);
      ow[k] = pack_bf16(a0, a1);
    }
    stg_v8(out + 16 * q, ow);
  }
}

// Same arithmetic, but the 32 x 32 result block leaves through shared memory and two TMA tile stores (16 columns
// each, SWIZZLE_32B staging: 16-byte chunk index ^= (row >> 2) & 1, conflict-free for the row-per-lane writes).
// Row-per-thread st.global costs one L1 wavefront per lane per instruction; with the stores switched off a layer ran
// 8-22 % faster, although the bytes are few — the TMA path takes them off the LSU / L1.
__device__ __forceinline__ void epi_mul_tma(const TcParams& p, const RowInfo& r, int col, const uint32_t (&v)[32],
                                            const U8 (&g)[2], uint32_t stage, const CUtensorMap* tmo) {
  const int lane = threadIdx.x & 31;
  const uint32_t sw = (uint32_t)(lane >> 2) & 1u;
#pragma unroll
  for (int q = 0; q < 2; ++q) {
    uint32_t ow[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      float a0 = __uint_as_float(v[16 * q + 2 * k]) * bf16_lo(g[q].w[k]);
      float a1 = __uint_as_float(v[16 * q + 2 * k + 1]) * bf16_hi(g[q].w[k]);
      ow[k] = r.valid ? pack_bf16(a0, a1) : 0u;          // padding rows of the PF layout stay exactly zero
    }
    if (lane == 0) bulk_wait_read0();                    // the previous store has finished reading the staging block
    __syncwarp();
    const uint32_t row_addr = stage + (uint32_t)lane * 32u;
    sts_v4(row_addr + ((0u ^ sw) << 4), ow[0], ow[1], ow[2], ow[3]);
    sts_v4(row_addr + ((1u ^ sw) << 4), ow[4], ow[5], ow[6], ow[7]);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncwarp();
    if (lane == 0) {
      tma_store_2d(tmo, stage, col + 16 * q, r.row - lane);
      bulk_commit();
    }
  }
}

// tile at pooled resolution; 16 columns starting at `col`: scatter to the 2x2 fine pixels chosen by the argmax bytes
// (the other three get 0).  g = 16 gains (bf16), sidx = 16 argmax bytes.
// 16-bit lane masks of "argmax byte == k" for the four channels of one pool_idx word (bytes 0..3 = channels 4i..4i+3):
// m01 covers the bf16 pair (4i, 4i+1), m23 the pair (4i+2, 4i+3).  0x80 - (byte ^ k) has its top bit set iff the byte equals
// k (bytes limited to 7 bits by the caller: no borrow between bytes), and PRMT's sign-replicate mode widens that bit to a
// half-word: 4 instructions per pool_idx word and k where the compare / select form took ~16 — the un-pool epilogue
// ran 1111 instructions per 32 x 32 unit, half of them this selection, and the layer is bound by instruction issue
// (profiles/r2_unpool_layer.md, DESIGN.md section 7).
__device__ __forceinline__ void unpool_masks(uint32_t idx7 /* pool_idx word & 0x7F7F7F7F */, uint32_t k, uint32_t& m01,
                                             uint32_t& m23) {
  const uint32_t s = 0x80808080u - (idx7 ^ (k * 0x01010101u));
  // (inline PTX: the __byte_perm intrinsic documents only the low three bits of a selector nibble)
  asm("prmt.b32 %0, %1, %1, 0x9988;" : "=r"(m01) : "r"(s));
  asm("prmt.b32 %0, %1, %1, 0xBBAA;" : "=r"(m23) : "r"(s));
}

__device__ __forceinline__ void epi_mul_unpool16(const TcParams& p, const RowInfo& r, int col, const uint32_t (&v)[16],
                                                 const U8& g, const uint4& sidx) {
  if (!r.in_range) return;
  const int wf1 = 2 * p.w + 1;
  const long long blk_f = (long long)(2 * p.h + 1) * wf1;
  // fine pixel (2a-1, 2b-1) of this pooled pixel; the other three are one pixel to the right / one fine row down.  Row -1
  // (a == 0) and column -1 (b == 0) do not exist: those stores are skipped, the pointer is never dereferenced.
  __nv_bfloat16* const p00 = reinterpret_cast<__nv_bfloat16*>(p.out) +
                             ((long long)r.e * blk_f + (long long)(2 * r.a - 1) * wf1 + (2 * r.b - 1)) * p.out_c + col;
  uint32_t prod[8];   // bf16x2 products: prod[j] = channels 2j, 2j+1
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    float a0 = __uint_as_float(v[2 * k]) * bf16_lo(g.w[k]);
    float a1 = __uint_as_float(v[2 * k + 1]) * bf16_hi(g.w[k]);
    prod[k] = r.valid ? pack_bf16(a0, a1) : 0u;
  }
  const uint32_t sw[4] = {sidx.x & 0x7F7F7F7Fu, sidx.y & 0x7F7F7F7Fu, sidx.z & 0x7F7F7F7Fu, sidx.w & 0x7F7F7F7Fu};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const bool ok = ((k >> 1) || r.a > 0) && ((k & 1) || r.b > 0);
    uint32_t ow[8];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t m01, m23;
      unpool_masks(sw[i], (uint32_t)k, m01, m23);
      ow[2 * i] = prod[2 * i] & m01;
      ow[2 * i + 1] = prod[2 * i + 1] & m23;
    }
    if (ok) stg_v8(p00 + ((long long)(k >> 1) * wf1 + (k & 1)) * p.out_c, ow);
  }
}

// forward + gain, 16 output channels starting at `ch`: vw = acc of W, vp = acc of W+
__device__ __forceinline__ void epi_fwd_gain16(const TcParams& p, const RowInfo& r, int ch, const uint32_t (&vw)[16],
                                               const uint32_t (&vp)[16]) {
  if (!r.in_range) return;
  __nv_bfloat16* act = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)r.row * p.out_c + ch;
  __nv_bfloat16* gn = reinterpret_cast<__nv_bfloat16*>(p.out2) + (size_t)r.row * p.out_c + ch;
  if (!r.valid) {
    stg_zero32(act);
    stg_zero32(gn);
    return;
  }
  // the bias of the 16 channels as four 16-byte loads; the quotient goes to bf16 (8 mantissa bits), so the
  // approximate division (MUFU.RCP + FMUL, 2 ulp) replaces the ~20-instruction IEEE sequence: with the IEEE form
  // this epilogue, not the tensor pipe, bounded every forward layer with K <= 1152 (measured)
  float bv[16];
  if (p.bias) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(p.bias + ch) + q);
      bv[4 * q] = t.x; bv[4 * q + 1] = t.y; bv[4 * q + 2] = t.z; bv[4 * q + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int q = 0; q < 16; ++q) bv[q] = 0.f;
  }
  const bool unit_num = p.gain_mode != 0;
  uint32_t aw[8], gw[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float a0 = fmaxf(__uint_as_float(vw[2 * k]) + bv[2 * k], 0.f);
    const float a1 = fmaxf(__uint_as_float(vw[2 * k + 1]) + bv[2 * k + 1], 0.f);
    float zp0 = __uint_as_float(vp[2 * k]), zp1 = __uint_as_float(vp[2 * k + 1]);
    zp0 += (zp0 == 0.f ? LRPX_Z_EPSILON : 0.f);          // safe_divide, utils.py:16-18
    zp1 += (zp1 == 0.f ? LRPX_Z_EPSILON : 0.f);
    const float g0 = __fdividef(unit_num ? 1.f : a0, zp0), g1 = __fdividef(unit_num ? 1.f : a1, zp1);
    aw[k] = pack_bf16(a0, a1);
    gw[k] = pack_bf16(g0, g1);
  }
  stg_v8(act, aw);
  stg_v8(gn, gw);
}

// first layer: acc columns 0..2 = W+^T s, 3..5 = W-^T s  ->  fp32 NCHW heat-map
__device__ __forceinline__ void epi_input(const TcParams& p, const RowInfo& r, const uint32_t (&v)[16]) {
  if (!r.valid) return;
  int img = p.row_img ? p.row_img[r.e] : r.e;
  size_t hw = (size_t)p.h * p.w;
  size_t pix = (size_t)(r.a - 1) * p.w + (r.b - 1);
  float* out = reinterpret_cast<float*>(p.out);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float xv = __ldg(p.x + ((size_t)img * 3 + c) * hw + pix);
    out[((size_t)r.e * 3 + c) * hw + pix] =
        fmaxf(xv, 0.f) * __uint_as_float(v[c]) + fminf(xv, 0.f) * __uint_as_float(v[3 + c]);
  }
}

// release_bar != 0 (the warp's LAST unit of the tile): the accumulator buffer is handed back to the MMA issuers as
// soon as this warp's last TMEM read has landed in registers, i.e. before the epilogue math and the global stores —
// the stores are the slow part of the epilogue (measured: 8-22 % of a layer's time) and must not sit on the
// TMEM hand-over path.
// pair mode (tcgen05.mma.cta_group::2): the accumulators of BOTH CTAs are written by the leader's MMAs, so the peer's
// epilogue warps hand their buffer back on the LEADER's barrier (release_bar is then a shared::cluster address)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void epi_release(const TcParams& p, uint32_t release_bar) {
  if (release_bar) {
    tc_fence_before();
    __syncwarp();
    if ((threadIdx.x & 31) == 0) {
      if (p.pair) mbar_arrive_cluster(release_bar);
      else mbar_arrive(release_bar);
    }
  }
}

// First layer with the three filter COLUMNS folded into N (LRPX_TC_EPI_INPUT3).  The N = 16 form issues 36 MMAs per 128
// rows and every one of them is bound by its 4 KB A read from shared memory (~46 cycles instead of 8): the layer runs at
// 1/6 of what its bytes allow.  Here one MMA chain per filter ROW (A view shifted by (dy-1)(w+1) rows, no column shift)
// produces P'[q][dx*8 + c] = sum_{dy,ch} s[q + (dy-1)(w+1)][ch] W[c][dy,dx][ch]  (c < 3: W+, 3..5: W-), 12 MMAs per 128
// rows, and the column shift moves to the epilogue:  acc[p][c] = P'[p-1][0,c] + P'[p][1,c] + P'[p+1][2,c].
// Neighbouring rows are neighbouring TMEM lanes = neighbouring threads: warp shuffles, plus a 48-byte exchange through
// shared memory at the three warp boundaries of a 128-row block.  The first and last row of a block have no neighbour,
// so the M halves of a tile start 126 rows apart and a tile yields 252 output rows.
template <bool CAM>
__device__ __forceinline__ void epi_input3(const TcParams& p, const RowInfo& r, uint32_t taddr, uint32_t release_bar,
                                           float* scratch /* [4 quarters][2][8] of this (buffer, half) */, int quarter,
                                           int bar_id, uint32_t full_bar, uint32_t full_parity) {
  const int lane = threadIdx.x & 31;
  const bool edge = (quarter == 0 && lane == 0) || (quarter == 3 && lane == 31);
  const bool writes = r.valid && !edge && !(p.debug_flags & 1);
  // the three input values of this pixel: issued before the accumulator read so that their L2 latency hides under it
  const int img = p.row_img ? p.row_img[r.e] : r.e;
  const size_t hw = (size_t)p.h * p.w;
  const size_t pix = writes ? (size_t)(r.a - 1) * p.w + (r.b - 1) : 0;
  float xin[3] = {0.f, 0.f, 0.f};
  if (writes)
#pragma unroll
    for (int c = 0; c < 3; ++c) xin[c] = __ldg(p.x + ((size_t)img * 3 + c) * hw + pix);
  // Guided Grad-CAM: this pixel's factor (Kw cam_rows^T)[y][x], formed in lrpx_cam_expand_mul_f32's fmaf order; its loads
  // and sum run, like the input values', before the accumulator wait
  float cam_v = 1.f;
  if (CAM && writes) {
    const float* t = p.cam_rows + ((size_t)r.e * p.h + (r.a - 1)) * p.cam_w;
    const float* kw = p.cam_kw + (size_t)(r.b - 1) * p.cam_w;
    cam_v = 0.f;
    for (int j = 0; j < p.cam_w; ++j) cam_v = fmaf(__ldg(kw + j), __ldg(t + j), cam_v);
  }
  // only now wait for the tile's accumulator: the row arithmetic and the two dependent loads above (request -> image, image
  // -> pixel values) used to start AFTER the wait and sat, with the integer divisions of tile_coords, on the pass's critical
  // path — the layer's tile time is the latency of one such pass (two warp sets alternate), not its bytes or its MMAs
  mbar_wait_ns(full_bar, full_parity, (uint32_t)p.sleep_ns);
  tc_fence_after();
  uint32_t v[24];
  TMEM_LD_X16(taddr, v);
  {
    uint32_t (&v8)[8] = *reinterpret_cast<uint32_t (*)[8]>(&v[16]);
    TMEM_LD_X8(taddr + 16, v8);
  }
  tmem_ld_wait();
  epi_release(p, release_bar);
  float up[6], dn[6];
#pragma unroll
  for (int c = 0; c < 6; ++c) {
    up[c] = __shfl_up_sync(0xffffffffu, __uint_as_float(v[c]), 1);          // P'[q-1][dx = 0]
    dn[c] = __shfl_down_sync(0xffffffffu, __uint_as_float(v[16 + c]), 1);   // P'[q+1][dx = 2]
  }
  if (lane == 0)
#pragma unroll
    for (int c = 0; c < 6; ++c) scratch[(quarter * 2 + 0) * 8 + c] = __uint_as_float(v[16 + c]);
  if (lane == 31)
#pragma unroll
    for (int c = 0; c < 6; ++c) scratch[(quarter * 2 + 1) * 8 + c] = __uint_as_float(v[c]);
  // the four quarter warps of this M half meet on their own named barrier (immediate ids: ptxas counts them)
  if (bar_id == 1) asm volatile("bar.sync 1, 128;" ::: "memory");
  else if (bar_id == 2) asm volatile("bar.sync 2, 128;" ::: "memory");
  else if (bar_id == 3) asm volatile("bar.sync 3, 128;" ::: "memory");
  else asm volatile("bar.sync 4, 128;" ::: "memory");
  if (lane == 0 && quarter > 0)
#pragma unroll
    for (int c = 0; c < 6; ++c) up[c] = scratch[((quarter - 1) * 2 + 1) * 8 + c];
  if (lane == 31 && quarter < 3)
#pragma unroll
    for (int c = 0; c < 6; ++c) dn[c] = scratch[((quarter + 1) * 2 + 0) * 8 + c];
  if (!writes) return;
  float res[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float xv = xin[c];
    const float cp = up[c] + __uint_as_float(v[8 + c]) + dn[c];
    const float cn = up[3 + c] + __uint_as_float(v[8 + 3 + c]) + dn[3 + c];
    // rules 2 / 3 (gradient family): the gradient with respect to the image itself, no multiplication by x
    res[c] = p.rule >= 2 ? cp : fmaxf(xv, 0.f) * cp + fminf(xv, 0.f) * cn;
  }
  // a rounded product (never contracted into the channel mean's additions): the same value lrpx_cam_expand_mul_f32 stores
  if (CAM)
#pragma unroll
    for (int c = 0; c < 3; ++c) res[c] = __fmul_rn(res[c], cam_v);
  // delivery format (gain_mode): 0 = fp32 (Q,3,h,w), the reference's return value; 1 = channel mean fp32 (Q,h,w) — what
  // every consumer in evaluation.py reduces a heat-map to first (:134,:411,:503: torch.mean(relevance, dim=(0,1)));
  // 2 = fp16 (Q,3,h,w)
  if (p.gain_mode == 1) {
    reinterpret_cast<float*>(p.out)[(size_t)r.e * hw + pix] = ((res[0] + res[1]) + res[2]) / 3.f;
  } else if (p.gain_mode == 2) {
    __half* out = reinterpret_cast<__half*>(p.out);
#pragma unroll
    for (int c = 0; c < 3; ++c) out[((size_t)r.e * 3 + c) * hw + pix] = __float2half_rn(res[c]);
  } else {
    float* out = reinterpret_cast<float*>(p.out);
#pragma unroll
    for (int c = 0; c < 3; ++c) out[((size_t)r.e * 3 + c) * hw + pix] = res[c];
  }
}

// ------------------------------------------------------------------------------------------ general epilogues
// value pair -> bf16x2 of the high parts and bf16x2 of the residuals (v = hi + lo to 16 significant bits)
__device__ __forceinline__ void split_pack(float v0, float v1, uint32_t& hi, uint32_t& lo) {
  hi = pack_bf16(v0, v1);
  lo = pack_bf16(v0 - bf16_lo(hi), v1 - bf16_hi(hi));
}
// 16 gains starting at element offset `off`: bf16 (32 bytes) or fp32 (64 bytes)
__device__ __forceinline__ void load_gain16(const void* base, size_t off, bool f32, float (&g)[16]) {
  if (f32) {
    const U8 a = ldg_nc_v8(reinterpret_cast<const float*>(base) + off);
    const U8 b = ldg_nc_v8(reinterpret_cast<const float*>(base) + off + 8);
#pragma unroll
    for (int k = 0; k < 8; ++k) { g[k] = __uint_as_float(a.w[k]); g[8 + k] = __uint_as_float(b.w[k]); }
  } else {
    const U8 a = ldg_nc_v8(reinterpret_cast<const __nv_bfloat16*>(base) + off);
#pragma unroll
    for (int k = 0; k < 8; ++k) { g[2 * k] = bf16_lo(a.w[k]); g[2 * k + 1] = bf16_hi(a.w[k]); }
  }
}

// MULX / MULX_UNPOOL: 32 accumulator columns [c, c+32) of this thread's row as two halves of 16.
//   group j:  v = acc * gain_j  ->  out[row][j*N + n] (hi)  and, when split, out[row][(G+j)*N + n] (lo)
// UNPOOL: the row is a pooled pixel; the products go to the winner of its 2x2 fine block, zeros to the other three.
// SIMPLE: one gain group, no residual addend, no second output tensor (every layer of a VGG-style chain in the
// fp32-accurate / gradient modes) — instantiated on its own (TC_EPI_MULX_S / TC_EPI_MULX_UNPOOL_S) so that the group loop
// and the fork state of the general form do not cost it registers (the general un-pool epilogue spills 160-200 bytes).
template <bool UNPOOL, bool SIMPLE>
__device__ __forceinline__ void epi_mulx(const TcParams& p, const RowInfo& r, uint32_t taddr, int n0, int c,
                                         uint32_t release_bar) {
  const int N = p.ncol, G = SIMPLE ? 1 : p.groups;
  const bool sp = p.split != 0;
  const int img = (r.valid && p.row_img) ? p.row_img[r.e] : r.e;
  const size_t gbase = ((size_t)img * p.blk + r.rem) * (size_t)N;
  __nv_bfloat16* const out = reinterpret_cast<__nv_bfloat16*>(p.out);
#pragma unroll 1
  for (int q = 0; q < 2; ++q) {
    const int col = n0 + c + 16 * q;
    float g[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) g[k] = 0.f;
    uint4 sidx = make_uint4(0u, 0u, 0u, 0u);          // pool_idx == nullptr: every winner is the window's first pixel
    if (r.valid) {
      load_gain16(p.gain, gbase + col, sp, g);
      if (UNPOOL && p.pool_idx) sidx = ldg_nc_v4(p.pool_idx + gbase + col);
    }
    uint32_t v[16];
    TMEM_LD_X16(taddr + c + 16 * q, v);
    tmem_ld_wait();
    if (q == 1) epi_release(p, release_bar);
    if (!r.in_range) continue;
#pragma unroll 1
    for (int j = 0; j < G; ++j) {
      if (j == 1 && r.valid) load_gain16(p.gain2, gbase + col, sp, g);
      float t[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) t[k] = 0.f;
      if (!SIMPLE && !UNPOOL && p.add && r.valid) {      // fork of a residual block: the other branch's relevance joins here
        float ad[16], gb[16];
        load_gain16(p.add, (size_t)r.row * p.add_pitch + col, false, ad);
        const void* gbp = j ? p.gain4 : p.gain3;           // nullptr: the addend joins unscaled
        if (gbp) load_gain16(gbp, gbase + col, sp, gb);
        else {
#pragma unroll
          for (int k = 0; k < 16; ++k) gb[k] = 1.f;
        }
#pragma unroll
        for (int k = 0; k < 16; ++k) t[k] = ad[k] * gb[k];
      }
      uint32_t hi[8], lo[8];
      // rule 3 (guided backpropagation, gridTDmodel.py:1680-1686): only the positive part of the incoming gradient
      // passes a ReLU
      const bool guided = p.rule == 3;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        float v0 = __uint_as_float(v[2 * k]), v1 = __uint_as_float(v[2 * k + 1]);
        if (guided) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
        const float a0 = r.valid ? fmaf(v0, g[2 * k], t[2 * k]) : 0.f;
        const float a1 = r.valid ? fmaf(v1, g[2 * k + 1], t[2 * k + 1]) : 0.f;
        split_pack(a0, a1, hi[k], lo[k]);
      }
      if (!UNPOOL) {
        if (!SIMPLE && j == 1 && p.out2) {    // two separate tensors instead of one K-concatenated row
          stg_v8(reinterpret_cast<__nv_bfloat16*>(p.out2) + (size_t)r.row * N + col, hi);
        } else {
          __nv_bfloat16* dst = out + (size_t)r.row * p.out_c + col;
          stg_v8(dst + (size_t)j * N, hi);
          if (sp) stg_v8(dst + (size_t)(G + j) * N, lo);
        }
      } else {
        const int wf1 = 2 * p.w + 1;
        const size_t blk_f = (size_t)(2 * p.h + 1) * wf1;
        __nv_bfloat16* const outb = out + (size_t)r.e * blk_f * p.out_c + col;
        const uint32_t sw[4] = {sidx.x, sidx.y, sidx.z, sidx.w};
#pragma unroll 1          // one fine pixel at a time: unrolled, the four address chains pushed the epilogue into 200 B of spills
        for (int k = 0; k < 4; ++k) {
          const int fr = 2 * r.a - 1 + (k >> 1), fc = 2 * r.b - 1 + (k & 1);
          if (fr < 0 || fc < 0) continue;
          __nv_bfloat16* dst = outb + ((size_t)fr * wf1 + fc) * p.out_c;
          uint32_t oh[8], ol[8];
#pragma unroll
          for (int m = 0; m < 4; ++m) {
            uint32_t m01, m23;
            unpool_masks(sw[m] & 0x7F7F7F7Fu, (uint32_t)k, m01, m23);
            oh[2 * m] = hi[2 * m] & m01;
            ol[2 * m] = lo[2 * m] & m01;
            oh[2 * m + 1] = hi[2 * m + 1] & m23;
            ol[2 * m + 1] = lo[2 * m + 1] & m23;
          }
          stg_v8(dst + (size_t)j * N, oh);
          if (sp) stg_v8(dst + (size_t)(G + j) * N, ol);
        }
      }
    }
  }
}

__device__ __forceinline__ void stg_f32x16(float* dst, const float (&v)[16]) {
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    uint32_t w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = __float_as_uint(v[8 * h + k]);
    stg_v8(dst + 8 * h, w);
  }
}

// FWDX: 32 output channels [c, c+32) of tile column block n_tile (see LRPX_TC_EPI_FWDX in lrpx.h)
__device__ __forceinline__ void load_bf16x16(const void* base, size_t off, float (&g)[16]) {
  const U8 a = ldg_nc_v8(reinterpret_cast<const __nv_bfloat16*>(base) + off);
#pragma unroll
  for (int k = 0; k < 8; ++k) { g[2 * k] = bf16_lo(a.w[k]); g[2 * k + 1] = bf16_hi(a.w[k]); }
}
__device__ __forceinline__ void store_act16(void* base, size_t off, size_t lo_off, bool sp, const float (&v)[16]) {
  uint32_t hi[8], lo[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) split_pack(v[2 * k], v[2 * k + 1], hi[k], lo[k]);
  __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(base) + off;
  stg_v8(dst, hi);
  if (sp) stg_v8(dst + lo_off, lo);
}
__device__ __forceinline__ void store_gain16(void* base, size_t off, bool f32, const float (&v)[16]) {
  if (f32) {
    stg_f32x16(reinterpret_cast<float*>(base) + off, v);
  } else {
    uint32_t w[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) w[k] = pack_bf16(v[2 * k], v[2 * k + 1]);
    stg_v8(reinterpret_cast<__nv_bfloat16*>(base) + off, w);
  }
}

// FWDX for a VGG-style layer (p.fwd_simple): act = relu(acc_W + bias), ONE gain group — alpha * num / safe(acc_W+)
// (rule 0), num' / stab(acc_W) (rule 1) or [act > 0] (rules 2 / 3).  Same arithmetic as epi_fwdx below, without the
// BatchNorm / Add / strided-store / extra-output state, whose registers made the general form spill 350 bytes per thread:
// the fp32-accurate forward of VGG16 ran at a sixth of its bf16 speed because of that.
__device__ __forceinline__ void epi_fwdx_simple(const TcParams& p, const RowInfo& r, uint32_t taddr, int n_tile, int c,
                                                uint32_t release_bar) {
  const bool sp = p.split != 0;
  const int cout = p.cout;
  // one unit = 16 output channels (epi_units_per_half): a 64-channel layer then keeps all four warps of a lane quarter
  // busy (with 32-column units two of them had nothing to do and the other two ran two serial passes)
  {
    const int ch = n_tile * p.half + c;
    uint32_t vw[16], vp[16];
    TMEM_LD_X16(taddr + c, vw);
    if (p.n_acc >= 2) TMEM_LD_X16(taddr + p.half + c, vp);
    tmem_ld_wait();
    epi_release(p, release_bar);
    if (!r.in_range) return;
    float bv[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) bv[k] = 0.f;
    if (p.bias) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p.bias + ch) + k4);
        bv[4 * k4] = t.x; bv[4 * k4 + 1] = t.y; bv[4 * k4 + 2] = t.z; bv[4 * k4 + 3] = t.w;
      }
    }
    float act[16], g0[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float zw = __uint_as_float(vw[k]);
      const float a = r.valid ? fmaxf(zw + bv[k], 0.f) : 0.f;
      act[k] = a;
      const float num = p.gain_mode ? 1.f : a;
      float q0;
      // gains as numerator x correctly-rounded reciprocal (<= 1.5 ulp off the IEEE quotient).  The IEEE division's
      // fast path rejects a zero dividend — half of the post-ReLU numerators — and a warp with ONE such lane runs the
      // slow-path subroutine for all 16 elements with its registers spilled to local memory (L1 is ~28 KB next to the
      // 200 KB of shared memory): measured 6.5 M slow-path calls per layer-0 launch, 2.5 ms instead of ~1 ms
      if (p.rule == 0) {
        float zp = __uint_as_float(vp[k]) + (p.zbias ? bv[k] : 0.f);
        zp += (zp == 0.f ? LRPX_Z_EPSILON : 0.f);
        q0 = p.alpha * num * __frcp_rn(zp);
      } else if (p.rule == 1) {
        const float zr = zw + (p.zbias ? bv[k] : 0.f);
        const float nq = (num == 0.f) ? -1e-6f : num;
        q0 = nq * __frcp_rn(p.zbias ? zr : stab(zr));
      } else {
        q0 = a > 0.f ? 1.f : 0.f;
      }
      g0[k] = r.valid ? q0 : 0.f;
    }
    const size_t go = (size_t)r.row * cout + ch;
    store_act16(p.out, (size_t)r.row * (size_t)(cout * (sp ? 2 : 1)) + ch, cout, sp, act);
    store_gain16(p.out2, go, sp, g0);
  }
}

// SPLIT_ADD: the residual operands of the fp32-accurate (split) forward, instantiated on its own (TC_EPI_FWDX_SPLIT_ADD)
// so that the bf16 form keeps its registers and spills
template <bool SPLIT_ADD>
__device__ __forceinline__ void epi_fwdx(const TcParams& p, const RowInfo& r, uint32_t taddr, int n_tile, int c,
                                         uint32_t release_bar) {
  const bool sp = p.split != 0;
  const int cout = p.cout;
  // strided store (fwd_flags bit 1): a stride-2 convolution is the stride-1 result at the even pixels; only those rows
  // are written, into a PF tensor of half the resolution (whose padding rows the caller has zeroed)
  const bool sub2 = (p.fwd_flags & 2) != 0;
  bool store = r.in_range;
  size_t orow = (size_t)r.row;
  if (sub2) {
    store = r.valid && ((r.a - 1) & 1) == 0 && ((r.b - 1) & 1) == 0;
    const int hc = p.h >> 1, wc = p.w >> 1;
    orow = (size_t)r.e * (size_t)((hc + 1) * (wc + 1)) + (size_t)(((r.a - 1) >> 1) + 1) * (wc + 1) + (((r.b - 1) >> 1) + 1);
  }
#pragma unroll 1
  for (int q = 0; q < 2; ++q) {
    const int ch = n_tile * p.half + c + 16 * q;
    uint32_t vw[16], vp[16], vn[16];
    TMEM_LD_X16(taddr + c + 16 * q, vw);
    if (p.n_acc >= 2) TMEM_LD_X16(taddr + p.half + c + 16 * q, vp);
    if (p.n_acc >= 3) TMEM_LD_X16(taddr + 2 * p.half + c + 16 * q, vn);
    tmem_ld_wait();
    if (q == 1) epi_release(p, release_bar);
    if (!store) continue;
    float bv[16], sw[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) { bv[k] = 0.f; sw[k] = 1.f; }
    const float* shift = p.bn_w ? p.bn_b : p.bias;
    if (shift) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(shift + ch) + k4);
        bv[4 * k4] = t.x; bv[4 * k4 + 1] = t.y; bv[4 * k4 + 2] = t.z; bv[4 * k4 + 3] = t.w;
      }
    }
    if (p.bn_w) {
#pragma unroll
      for (int k4 = 0; k4 < 4; ++k4) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(p.bn_w + ch) + k4);
        sw[4 * k4] = t.x; sw[4 * k4 + 1] = t.y; sw[4 * k4 + 2] = t.z; sw[4 * k4 + 3] = t.w;
      }
    }
    float idv[16], hdv[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) { idv[k] = 0.f; hdv[k] = 1.f; }
    const size_t go = orow * cout + ch;
    if (SPLIT_ADD) {
      // idn is a hi|lo row of 2*cout (its value hi + lo; hdv holds lo for the moment), hd an fp32 gain (store_gain16, split)
      if (p.idn && r.valid) {
        load_bf16x16(p.idn, orow * (2 * cout) + ch, idv);
        load_bf16x16(p.idn, orow * (2 * cout) + cout + ch, hdv);
#pragma unroll
        for (int k = 0; k < 16; ++k) { idv[k] += hdv[k]; hdv[k] = 1.f; }
      }
      if (p.hd && r.valid) load_gain16(p.hd, go, true, hdv);
    } else {
      if (p.idn && r.valid) load_bf16x16(p.idn, go, idv);
      if (p.hd && r.valid) load_bf16x16(p.hd, go, hdv);
    }
    float act[16], g0[16], g1[16], ag0[16], ag1[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float zw = __uint_as_float(vw[k]);
      const float y = fmaf(zw, sw[k], bv[k]);                        // conv + bias, or the folded BatchNorm
      const float o = y + idv[k];                                    // residual Add (resnet.py:33-38)
      const float a = r.valid ? ((p.fwd_flags & 1) ? o : fmaxf(o, 0.f)) : 0.f;
      act[k] = a;
      // BatchNorm rule (lrp_modules.py:204-215): R = |x w| / (|x w| + |b|) R_out, safe_divide
      float ratio = 1.f;
      if (p.bn_w) {
        const float xw = fabsf(zw * sw[k]), den = xw + fabsf(bv[k]);
        ratio = xw / (den + (den == 0.f ? LRPX_Z_EPSILON : 0.f));
      }
      // Add rule (lrp_modules.py:262-275): x_i / (out + 0.01 sign out); out == 0 -> 0.5 each
      float rho1 = 1.f, rho2 = 0.f;
      if (p.idn) {
        if (o == 0.f) { rho1 = 0.5f; rho2 = 0.5f; }
        else { const float so = o + (o > 0.f ? 0.01f : -0.01f); rho1 = y / so; rho2 = idv[k] / so; }
      }
      const float num = p.gain_mode ? 1.f : a;
      float q0 = 0.f, q1 = 0.f;
      if (p.rule == 0) {
        float zp = __uint_as_float(vp[k]) + (p.zbias ? bv[k] : 0.f);
        zp += (zp == 0.f ? LRPX_Z_EPSILON : 0.f);                   // safe_divide, utils.py:16-18
        q0 = p.alpha * num * ratio * rho1 * __frcp_rn(zp);           // reciprocal, not division: see epi_fwdx_simple
        if (p.n_acc >= 3) {
          float zn = __uint_as_float(vn[k]) + (p.zbias ? bv[k] : 0.f);
          zn += (zn == 0.f ? LRPX_Z_EPSILON : 0.f);
          q1 = -p.beta * num * __frcp_rn(zn);
        } else if (p.idn) {
          q1 = rho2 * hdv[k];                                        // identity-branch gain
        }
      } else if (p.rule == 1) {
        const float zr = zw + (p.zbias ? bv[k] : 0.f);
        const float nq = (num == 0.f) ? -1e-6f : num;               // zeros of the input count as -1e-6 (Q9)
        q0 = p.zbias ? nq / zr : nq / stab(zr);                     // the bias branch is unstabilised (lrp_modules.py:20-21)
      } else {
        q0 = a > 0.f ? 1.f : 0.f;                                   // rule 2 / 3: the ReLU's derivative (gradient family)
      }
      g0[k] = r.valid ? q0 : 0.f;
      g1[k] = r.valid ? q1 : 0.f;
      ag0[k] = a * g0[k];
      ag1[k] = a * g1[k];
    }
    store_act16(p.out, orow * (size_t)(cout * (sp ? 2 : 1)) + ch, cout, sp, act);
    store_gain16(p.out2, go, sp, g0);
    if (p.out3) store_gain16(p.out3, go, sp, g1);
    if (p.out4) store_gain16(p.out4, go, sp, ag0);
    if (p.out5) store_gain16(p.out5, go, sp, ag1);
  }
}

// MUL with folded filter columns (p.fold, 64 output channels): the tile's accumulator holds, per P' row q, three blocks of
// 64 columns   P'[q][dx, n] = sum_{dy, c} A[q + dy (w+1)][c] W[n][(dy, dx), c]   and the output row is
//   out[p][n] = gain[p][n] * (P'[p-1][0, n] + P'[p][1, n] + P'[p+1][2, n]).
// A 64-column MMA reads 4 KB of A and 2 KB of B from shared memory for 128 x 64 x 16 MACs and is bound by those reads
// (l1tex__data_pipe_tc_wavefronts_mem_shared 78 % at 52 % tensor-pipe activity, profiles/r2_chain_full.md); the folded form
// reads 4 + 6 KB for three times the MACs and a third of the MMAs.  Neighbouring rows are neighbouring TMEM lanes =
// neighbouring threads: warp shuffles, plus a 64-byte exchange through shared memory at the three warp boundaries of the
// 128-row tile; its first and last row have no neighbour, so a tile yields 126 output rows (as in epi_input3).
// One unit = 16 output channels [ch0, ch0 + 16): the four warps of a lane quarter take one unit each.
__device__ __forceinline__ void epi_mul_fold(const TcParams& p, const RowInfo& r, uint32_t taddr, int ch0,
                                             uint32_t release_bar, float* scratch /* [4 quarters][2][16] of this (buffer, unit) */,
                                             int quarter, int bar_id) {
  const int lane = threadIdx.x & 31;
  const int N = p.ncol;                                   // 64
  const bool edge = (quarter == 0 && lane == 0) || (quarter == 3 && lane == 31);
  U8 g;
#pragma unroll
  for (int k = 0; k < 8; ++k) g.w[k] = 0u;
  if (r.valid && !edge) {
    const int img = p.row_img ? p.row_img[r.e] : r.e;
    g = ldg_nc_v8(p.gain + ((size_t)img * p.blk + r.rem) * N + ch0);
  }
  uint32_t v0[16], v1[16], v2[16];
  TMEM_LD_X16(taddr + ch0, v0);
  TMEM_LD_X16(taddr + N + ch0, v1);
  TMEM_LD_X16(taddr + 2 * N + ch0, v2);
  tmem_ld_wait();
  epi_release(p, release_bar);
  float up[16], dn[16];
#pragma unroll
  for (int k = 0; k < 16; ++k) {
    up[k] = __shfl_up_sync(0xffffffffu, __uint_as_float(v0[k]), 1);       // P'[q-1][dx = 0]
    dn[k] = __shfl_down_sync(0xffffffffu, __uint_as_float(v2[k]), 1);     // P'[q+1][dx = 2]
  }
  if (lane == 0)
#pragma unroll
    for (int k = 0; k < 16; ++k) scratch[(quarter * 2 + 0) * 16 + k] = __uint_as_float(v2[k]);   // for the previous quarter's lane 31
  if (lane == 31)
#pragma unroll
    for (int k = 0; k < 16; ++k) scratch[(quarter * 2 + 1) * 16 + k] = __uint_as_float(v0[k]);   // for the next quarter's lane 0
  // the four quarter warps of this unit meet on their own named barrier (immediate ids: ptxas counts them)
  if (bar_id == 1) asm volatile("bar.sync 1, 128;" ::: "memory");
  else if (bar_id == 2) asm volatile("bar.sync 2, 128;" ::: "memory");
  else if (bar_id == 3) asm volatile("bar.sync 3, 128;" ::: "memory");
  else asm volatile("bar.sync 4, 128;" ::: "memory");
  if (lane == 0 && quarter > 0)
#pragma unroll
    for (int k = 0; k < 16; ++k) up[k] = scratch[((quarter - 1) * 2 + 1) * 16 + k];
  if (lane == 31 && quarter < 3)
#pragma unroll
    for (int k = 0; k < 16; ++k) dn[k] = scratch[((quarter + 1) * 2 + 0) * 16 + k];
  if (!r.in_range || edge || (p.debug_flags & 1)) return;
  uint32_t ow[8];
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    const float a0 = (up[2 * k] + __uint_as_float(v1[2 * k]) + dn[2 * k]) * bf16_lo(g.w[k]);
    const float a1 = (up[2 * k + 1] + __uint_as_float(v1[2 * k + 1]) + dn[2 * k + 1]) * bf16_hi(g.w[k]);
    ow[k] = r.valid ? pack_bf16(a0, a1) : 0u;             // padding rows are written as zeros
  }
  stg_v8(reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)r.row * N + ch0, ow);
}

// internal epilogue code (not part of the ABI): FWDX of a VGG-style layer, instantiated on its own so that the general
// FWDX epilogue's register pressure (BatchNorm / Add / strided-store state, 470 bytes of stack) stays out of it
constexpr int TC_EPI_FWDX_SIMPLE = 12;
constexpr int TC_EPI_MUL_FOLD = 15;         // MUL with the three filter COLUMNS folded into N (64-channel layers, epi_mul_fold)
constexpr int TC_EPI_MULX_S = 13, TC_EPI_MULX_UNPOOL_S = 14;      // MULX / MULX_UNPOOL with one gain group, no addend (epi_mulx)
constexpr int TC_EPI_FWDX_SPLIT_ADD = 16;   // FWDX with split rows and a residual operand (idn / hd): epi_fwdx<true>
constexpr int TC_EPI_INPUT3_CAM = 17;       // INPUT3 with Guided Grad-CAM's factor (cam_rows): epi_input3<true>, on its own so
                                            // that the factor's loop does not cost the plain first layer registers
__host__ __device__ constexpr bool is_input3(int epi) { return epi == LRPX_TC_EPI_INPUT3 || epi == TC_EPI_INPUT3_CAM; }

// number of 32-column units per (lane quarter, M half) of a tile
__device__ __forceinline__ int epi_units_per_half(const TcParams& p, int epi) {
  if (epi == LRPX_TC_EPI_INPUT || is_input3(epi)) return 1;
  if (epi == TC_EPI_MUL_FOLD) return 4;                   // four units of 16 output channels (`c` counts 32 per unit: c >> 1)
  if (epi == TC_EPI_FWDX_SIMPLE) return p.half >> 4;      // 16-column units (run_epilogue_tile: c = u << 4)
  const int ncols = (epi == LRPX_TC_EPI_FWD_GAIN || epi == LRPX_TC_EPI_FWDX || epi == TC_EPI_FWDX_SIMPLE ||
                     epi == TC_EPI_FWDX_SPLIT_ADD) ? p.half : p.bn;
  return ncols >> 5;
}

// One unit: accumulator row `r` (this thread's), columns [c, c+32) of tile column block n_tile.
// taddr = TMEM address of column 0 of this row's accumulator (lane quarter, buffer and M half already applied).
// Global loads of gain / argmax are issued first, then TMEM -> registers, epilogue math, global stores.
template <int EPI>
__device__ __forceinline__ void epi_unit(const TcParams& p, const RowInfo& r0, uint32_t taddr, int n_tile, int c,
                                         uint32_t release_bar, uint32_t stage = 0, const CUtensorMap* tmo = nullptr,
                                         float* scratch = nullptr, int quarter = 0, int bar_id = 0, uint32_t full_bar = 0,
                                         uint32_t full_parity = 0) {
  if (p.debug_flags & 16) {             // timing experiment: only hands the accumulator back
    if (is_input3(EPI)) { mbar_wait_ns(full_bar, full_parity, (uint32_t)p.sleep_ns); tc_fence_after(); }
    epi_release(p, release_bar);
    return;
  }
  RowInfo r = r0;
  if (p.debug_flags & 1) { r.in_range = false; r.valid = false; }
  const int n0 = n_tile * p.bn;
  if (is_input3(EPI)) {
    epi_input3<EPI == TC_EPI_INPUT3_CAM>(p, r, taddr, release_bar, scratch, quarter, bar_id, full_bar, full_parity);
  } else if (EPI == TC_EPI_MUL_FOLD) {
    epi_mul_fold(p, r0, taddr, c >> 1, release_bar, scratch, quarter, bar_id);
  } else if (EPI == LRPX_TC_EPI_MULX) {
    epi_mulx<false, false>(p, r, taddr, n0, c, release_bar);
  } else if (EPI == LRPX_TC_EPI_MULX_UNPOOL) {
    epi_mulx<true, false>(p, r, taddr, n0, c, release_bar);
  } else if (EPI == TC_EPI_MULX_S) {
    epi_mulx<false, true>(p, r, taddr, n0, c, release_bar);
  } else if (EPI == TC_EPI_MULX_UNPOOL_S) {
    epi_mulx<true, true>(p, r, taddr, n0, c, release_bar);
  } else if (EPI == TC_EPI_FWDX_SIMPLE) {
    epi_fwdx_simple(p, r, taddr, n_tile, c, release_bar);
  } else if (EPI == LRPX_TC_EPI_FWDX) {
    epi_fwdx<false>(p, r, taddr, n_tile, c, release_bar);
  } else if (EPI == TC_EPI_FWDX_SPLIT_ADD) {
    epi_fwdx<true>(p, r, taddr, n_tile, c, release_bar);
  } else if (EPI == LRPX_TC_EPI_INPUT) {
    uint32_t v[16];
    TMEM_LD_X16(taddr, v);
    tmem_ld_wait();
    epi_release(p, release_bar);
    epi_input(p, r, v);
  } else if (EPI == LRPX_TC_EPI_FWD_GAIN) {
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      uint32_t vw[16], vp[16];
      TMEM_LD_X16(taddr + c + 16 * q, vw);
      TMEM_LD_X16(taddr + p.half + c + 16 * q, vp);
      tmem_ld_wait();
      if (q == 1) epi_release(p, release_bar);
      epi_fwd_gain16(p, r, n_tile * p.half + c + 16 * q, vw, vp);
    }
  } else if (EPI == LRPX_TC_EPI_STORE_F32) {
    uint32_t v[32];
    TMEM_LD_X32(taddr + c, v);
    tmem_ld_wait();
    epi_release(p, release_bar);
    if (r.in_range && (p.fwd_flags & 4)) {
      // bf16 output (fwd_flags bit 2): halves the bytes of a GEMM whose result is only an intermediate (ResNet stem)
      __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.out) + (size_t)r.row * p.out_c + n0 + c;
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        uint32_t w[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) w[k] = pack_bf16(__uint_as_float(v[16 * q + 2 * k]), __uint_as_float(v[16 * q + 2 * k + 1]));
        stg_v8(dst + 16 * q, w);
      }
    } else if (r.in_range) {
      // out_c = row pitch, n_valid = columns that exist (a multiple of 4; the tile may be padded beyond it); the bias
      // (one value per column) turns the plain GEMM into a Linear layer
      const int col0 = n0 + c;
      float4* dst = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + (size_t)r.row * p.out_c + col0);
#pragma unroll
      for (int q = 0; q < 8; ++q) {
        if (col0 + 4 * q >= p.n_valid) break;
        float4 b4 = make_float4(0.f, 0.f, 0.f, 0.f);
        if (p.bias) b4 = __ldg(reinterpret_cast<const float4*>(p.bias + col0) + q);
        dst[q] = make_float4(__uint_as_float(v[4 * q]) + b4.x, __uint_as_float(v[4 * q + 1]) + b4.y,
                             __uint_as_float(v[4 * q + 2]) + b4.z, __uint_as_float(v[4 * q + 3]) + b4.w);
      }
    }
  } else if (EPI == LRPX_TC_EPI_FEAT || EPI == LRPX_TC_EPI_FEAT_DIV) {
    // rows = (request q = r.e, pixel p = r.rem); x / x1 are indexed by the request's image
    const int img = p.row_img ? p.row_img[r.e] : r.e;
    const size_t xo = ((size_t)img * p.blk + r.rem) * p.out_c + n0 + c;
    const size_t bo = (size_t)r.e * p.out_c + n0 + c;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      U8 xv[2], bv[2], dv[2];
#pragma unroll
      for (int k = 0; k < 8; ++k) bv[0].w[k] = bv[1].w[k] = 0u;
      if (r.in_range) {
        xv[0] = ldg_nc_v8(p.x + xo + 16 * q);
        xv[1] = ldg_nc_v8(p.x + xo + 16 * q + 8);
        if (p.bias) {
          bv[0] = ldg_nc_v8(p.bias + bo + 16 * q);
          bv[1] = ldg_nc_v8(p.bias + bo + 16 * q + 8);
        }
        if (EPI == LRPX_TC_EPI_FEAT_DIV) {
          dv[0] = ldg_nc_v8(p.x1 + xo + 16 * q);
          dv[1] = ldg_nc_v8(p.x1 + xo + 16 * q + 8);
        }
      }
      uint32_t v[16];
      TMEM_LD_X16(taddr + c + 16 * q, v);
      tmem_ld_wait();
      if (q == 1) epi_release(p, release_bar);
      if (r.in_range) {
        float* dst = reinterpret_cast<float*>(p.out) + (size_t)r.row * p.out_c + n0 + c + 16 * q;
#pragma unroll
        for (int hh = 0; hh < 2; ++hh) {
          uint32_t ow[8];
#pragma unroll
          for (int k = 0; k < 8; ++k) {
            float val = __uint_as_float(xv[hh].w[k]) * (__uint_as_float(v[8 * hh + k]) + __uint_as_float(bv[hh].w[k]));
            if (EPI == LRPX_TC_EPI_FEAT_DIV) val = val / stab(__uint_as_float(dv[hh].w[k]));
            ow[k] = __float_as_uint(val);
          }
          stg_v8(dst + 8 * hh, ow);
        }
      }
    }
  } else {   // MUL / MUL_UNPOOL
    size_t goff = 0;
    if (r.valid) {
      const int img = p.row_img ? p.row_img[r.e] : r.e;
      goff = ((size_t)img * p.blk + r.rem) * p.out_c + n0 + c;
    }
    U8 g[2];
    uint4 s4[2];
#pragma unroll
    for (int k = 0; k < 8; ++k) g[0].w[k] = g[1].w[k] = 0u;
    s4[0] = s4[1] = make_uint4(0u, 0u, 0u, 0u);
    if (r.valid && !(p.debug_flags & 32)) {      // 32: timing experiment without the gain loads
      g[0] = ldg_nc_v8(p.gain + goff);
      g[1] = ldg_nc_v8(p.gain + goff + 16);
      if (EPI == LRPX_TC_EPI_MUL_UNPOOL) {
        s4[0] = ldg_nc_v4(p.pool_idx + goff);
        s4[1] = ldg_nc_v4(p.pool_idx + goff + 16);
      }
    }
    if (EPI == LRPX_TC_EPI_MUL) {
      uint32_t v[32];
      TMEM_LD_X32(taddr + c, v);
      tmem_ld_wait();
      epi_release(p, release_bar);
      if (stage && !(p.debug_flags & 64)) epi_mul_tma(p, r, n0 + c, v, g, stage, tmo);
      else epi_mul(p, r, n0 + c, v, g);
    } else {
#pragma unroll
      for (int q = 0; q < 2; ++q) {
        uint32_t v[16];
        TMEM_LD_X16(taddr + c + 16 * q, v);
        tmem_ld_wait();
        if (q == 1) epi_release(p, release_bar);
        epi_mul_unpool16(p, r, n0 + c + 16 * q, v, g[q], s4[q]);
      }
    }
  }
}

// L2 prefetch of the gain (and argmax) bytes a unit will read, issued a couple of tiles ahead
template <int EPI>
__device__ __forceinline__ void epi_prefetch_unit(const TcParams& p, int row, int n_tile, int c) {
  constexpr bool simple_x = EPI == TC_EPI_MULX_S || EPI == TC_EPI_MULX_UNPOOL_S;
  if (EPI != LRPX_TC_EPI_MUL && EPI != LRPX_TC_EPI_MUL_UNPOOL && !simple_x) return;
  if (row >= p.m_total || (p.debug_flags & 128)) return;      // 128: timing experiment without the L2 prefetch
  const RowInfo q = row_info(p, row);
  if (!q.valid) return;
  const int img = p.row_img ? p.row_img[q.e] : q.e;
  if (simple_x) {                                             // gains of ncol channels per row, bf16 or fp32 (split)
    const size_t po = ((size_t)img * p.blk + q.rem) * (size_t)p.ncol + n_tile * p.bn + c;
    const char* g = reinterpret_cast<const char*>(p.gain) + po * (p.split ? 4 : 2);
    prefetch_l2(g);                                           // 32 columns: 64 bytes (bf16) or one 128-byte line (fp32)
    if (EPI == TC_EPI_MULX_UNPOOL_S && p.pool_idx) prefetch_l2(p.pool_idx + po);
    return;
  }
  const size_t po = ((size_t)img * p.blk + q.rem) * p.out_c + n_tile * p.bn + c;
  prefetch_l2(p.gain + po);                                   // 32 columns of bf16 = 64 bytes: one line
  if (EPI == LRPX_TC_EPI_MUL_UNPOOL) prefetch_l2(p.pool_idx + po);
}

// All units of one tile that belong to this epilogue warp.  sub = 0..3: which of the four warps of the lane quarter.
template <int EPI>
__device__ __forceinline__ void run_epilogue_tile(const TcParams& p, int row_base /* tile row 0 + quarter*32 + lane */,
                                                  uint32_t taddr_q /* lane quarter + buffer */, int n_tile, int sub,
                                                  int mh, int pf_row_base /* same for the prefetched tile, or -1 */,
                                                  uint32_t release_bar /* tmem_empty barrier of the tile's buffer */,
                                                  uint32_t stage = 0, const CUtensorMap* tmo = nullptr,
                                                  float* scratch = nullptr /* INPUT3: [2 halves][4][2][8] */, int quarter = 0,
                                                  int it = 0 /* this CTA's tile counter */,
                                                  uint32_t full_bar = 0 /* INPUT3: the caller has NOT waited for the */,
                                                  uint32_t full_parity = 0 /* accumulator yet (epi_input3 does) */) {
  const int uph = epi_units_per_half(p, EPI);
  const int n_units = mh * uph;
  constexpr int step = TC_EPI_WARPS / 4;
  // First-layer epilogues have only mh (<= 2) units per lane quarter, and a tile's MMAs are short: the tile time is the
  // LATENCY of one epilogue pass.  Warps 0,1 of a quarter therefore take the even tiles and warps 2,3 the odd ones, so
  // the passes of the two accumulator buffers overlap.
  int set = 0;
  if ((EPI == LRPX_TC_EPI_INPUT || is_input3(EPI)) && n_units <= 2) {
    set = it & 1;
    sub = set ? sub - 2 : sub;
    if (sub < 0 || sub >= 2) sub = n_units;          // not this warp's tile
  }
  if (sub >= n_units) {                 // nothing to read for this warp: hand the buffer back at once
    if (is_input3(EPI)) { mbar_wait_ns(full_bar, full_parity, (uint32_t)p.sleep_ns); tc_fence_after(); }
    epi_release(p, release_bar);
    return;
  }
  if (EPI == TC_EPI_MUL_FOLD) {         // one unit (16 output channels) per warp of the lane quarter
    const RowInfo rf = row_info(p, row_base);
    epi_unit<EPI>(p, rf, taddr_q, n_tile, sub << 5, release_bar, stage, tmo, scratch + sub * 128, quarter, 1 + sub);
    return;
  }
  int h_cached = -1;
  RowInfo r{};
  for (int u = sub; u < n_units; u += step) {
    const int h = u >= uph ? 1 : 0, c = (u - h * uph) << (EPI == TC_EPI_FWDX_SIMPLE ? 4 : 5);      // mh <= 2
    const int hr = (is_input3(EPI)) ? p.half_rows : TC_BM;
    if (h != h_cached) {
      r = row_info(p, row_base + h * hr);
      h_cached = h;
      // walk mode: the tiles are tile_stride (< tile_out_rows) rows apart; rows past the stride belong to the next tile
      if (is_input3(EPI) && p.walk && h * hr + quarter * 32 + (int)(threadIdx.x & 31) - p.fold >= p.tile_stride)
        r.valid = false;
    }
    if (pf_row_base >= 0) epi_prefetch_unit<EPI>(p, pf_row_base + h * TC_BM, n_tile, c);
    epi_unit<EPI>(p, r, taddr_q + (uint32_t)(h * p.bn), n_tile, c, (u + step >= n_units) ? release_bar : 0u, stage, tmo,
                  scratch ? scratch + h * 64 : nullptr, quarter, 1 + 2 * set + h, full_bar, full_parity);
  }
}

// ------------------------------------------------------------------------------------------ the kernel
template <int EPI>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_conv_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t full_bar[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t empty_bar[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t tmem_full_bar[2];
  __shared__ __align__(8) uint64_t tmem_empty_bar[2];
  __shared__ uint32_t tmem_base_slot;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // 1024-byte aligned tile ring (SWIZZLE_128B atoms are 1024 bytes)
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_bytes = (uint32_t)p.bn * TC_BK * 2;
  const uint32_t stage_bytes = TC_A_BYTES + b_bytes;
  const int num_tiles = p.num_m_tiles * p.num_n_tiles;
  const int num_kb = p.taps * p.kc_per_tap;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(smem_u32(&full_bar[s]), 1);
      mbar_init(smem_u32(&empty_bar[s]), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), 1);
      mbar_init(smem_u32(&tmem_empty_bar[b]), TC_EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                 "r"(512u)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_slot;

  if (warp == 0) {
    // ================================ TMA producer (one thread)
    if (elect_one()) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
        const int n_tile = tile % p.num_n_tiles, m_tile = tile / p.num_n_tiles;
        const int m0 = m_tile * TC_BM, n0 = n_tile * p.bn;
        for (int tap = 0; tap < p.taps; ++tap) {
          const int off = (p.taps == 9) ? ((tap / 3) - 1) * p.wp1 + ((tap % 3) - 1) : 0;
          for (int kc = 0; kc < p.kc_per_tap; ++kc) {
            mbar_wait_relaxed(smem_u32(&empty_bar[stage]), phase ^ 1);
            const uint32_t fb = smem_u32(&full_bar[stage]);
            const uint32_t sa = smem_base + stage * stage_bytes;
            mbar_expect_tx(fb, stage_bytes);
            const int kca = (p.a_wrap && kc >= p.a_wrap) ? kc - p.a_wrap : kc;      // hi | lo | hi view of a split row
            tma_load_2d(sa, &tmA, fb, kca * TC_BK, m0 + off);
            tma_load_2d(sa + TC_A_BYTES, &tmB, fb, tap * p.cin + kc * TC_BK, n0);
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ================================ MMA issuer (one thread)
    if (elect_one()) {
      const uint32_t idesc = make_idesc(p.bn);
      const uint32_t stage16 = stage_bytes >> 4;
      const uint32_t a_lo_base = desc_lo(smem_base), b_lo_base = desc_lo(smem_base + TC_A_BYTES);
      const int stages = p.stages;
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int buf = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(smem_u32(&tmem_empty_bar[buf]), acc_phase ^ 1);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + buf * 256;
        for (int kb = 0; kb < num_kb; ++kb) {
          mbar_wait(smem_u32(&full_bar[stage]), phase);
          tc_fence_after();
          const uint32_t a_lo = a_lo_base + (uint32_t)stage * stage16, b_lo = b_lo_base + (uint32_t)stage * stage16;
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k) {
            // advance 16 bf16 = 32 bytes along K inside the swizzle row: +2 in the (addr >> 4) field
            tc_mma_f16(d_tmem, desc_pack(a_lo + 2 * k), desc_pack(b_lo + 2 * k), idesc, (k == 0) ? (kb != 0 ? 1u : 0u) : 1u);
          }
          tc_commit(smem_u32(&empty_bar[stage]));       // frees the smem stage once these MMAs retire
          if (++stage == stages) { stage = 0; phase ^= 1; }
        }
        tc_commit(smem_u32(&tmem_full_bar[buf]));        // accumulator ready for the epilogue
      }
    }
  } else if (warp >= 2 && warp < 2 + TC_EPI_WARPS) {
    // ================================ epilogue warps
    const int quarter = warp & 3;
    int it = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
      const int buf = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      const int n_tile = tile % p.num_n_tiles, m_tile = tile / p.num_n_tiles;
      mbar_wait_relaxed(smem_u32(&tmem_full_bar[buf]), acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * 256;
      run_epilogue_tile<EPI>(p, m_tile * TC_BM + quarter * 32 + lane, taddr, n_tile, (warp - 2) >> 2, 1, -1,
                             smem_u32(&tmem_empty_bar[buf]));
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// tile index -> (M tile, N tile).  Cluster mode: the two CTAs of a pair (tile 2P, 2P+1) get the SAME column block and
// neighbouring M tiles, so they consume the same B tiles in the same order; m_tile may be one past the end (a padding
// tile: its A rows are zero-filled by TMA and its results are clipped by the row bound).
__device__ __forceinline__ void tile_coords(const TcParams& p, int tile, int& m_tile, int& n_tile) {
  // (host-prepared multiplier: the generic integer division is ~40 dependent instructions, twice per tile on every
  // epilogue warp's critical path — 8 % of the first layer's stall samples)
  if (p.cluster == 2) {
    const int pr = tile >> 1;
    const int q = fast_div(pr, p.nnt_mul, p.nnt_sh);
    n_tile = pr - q * p.num_n_tiles;
    m_tile = q * 2 + (tile & 1);
  } else {
    m_tile = fast_div(tile, p.nnt_mul, p.nnt_sh);
    n_tile = tile - m_tile * p.num_n_tiles;
  }
}

// MMA issue loop of the slab kernel.  Everything loop-invariant is hoisted and the taps x 4 K-steps are unrolled
// so that one MMA costs a handful of integer instructions (measured: ~200 cycles per MMA with the naive loop, which
// capped the N<=64 layers at 1/6 of the tensor rate; ~75 cycles with this loop and a converged issuing warp).
//
// Two issuer warps, in LOCKSTEP: with mh == 2 issuer j issues the MMAs of M half j (rows [128j, 128j+128) of the
// tile, TMEM columns [j*bn, (j+1)*bn) of the tile's accumulator buffer).  Both walk every tile, every A stage and
// every B tile in the same order; the a_empty / b_empty / tmem_full barriers count one tcgen05.commit per issuer,
// so neither issuer can run more than one ring revolution ahead of the other (mbarrier parity waits are only
// unambiguous one phase apart — giving the issuers alternate TILES on a shared ring is not safe).
// With mh == 1 only issuer 0 works (N = 256 MMAs occupy the tensor pipe for 128 cycles, one thread keeps up).
// PAIR: tcgen05.mma.cta_group::2 issued by the leader CTA of a pair for both (M = 256: this CTA's 128 rows and the same
// rows of the peer's slab at the same shared-memory offset; B: each CTA holds bn/2 rows of every tile); every commit
// arrives in both CTAs.
template <bool BRES, bool MODE3, int ISSUER, bool PAIR>
__device__ __forceinline__ void slab_mma_loop(const TcParams& p, uint64_t* a_full, uint64_t* a_empty, uint64_t* b_full,
                                              uint64_t* b_empty, uint64_t* bres_bar, uint64_t* tmem_full_bar,
                                              uint64_t* tmem_empty_bar, uint32_t a_base, uint32_t b_base,
                                              uint32_t tmem_base, int num_tiles) {
  // ISSUER is a template parameter (not a value derived from threadIdx) so that ptxas can prove every descriptor
  // warp-uniform and keep it in uniform registers
  constexpr int issuer = ISSUER;
  const uint32_t idesc = make_idesc(p.bn, PAIR ? 2 * TC_BM : TC_BM);
  // B tile pitch in 16-byte units (pair mode: each CTA stores its half tile at a half-size pitch)
  const uint32_t b16 = (((uint32_t)p.bn * TC_BK * 2) >> 4) >> (PAIR ? 1 : 0);
  const uint32_t a_stage16 = (uint32_t)p.a_stage_bytes >> 4;
  const uint32_t row16 = (TC_BK * 2) >> 4;                        // one PF row of 64 channels, 16-byte units
  // MODE3: each filter row has its own slab — a ring stage of its own, or (a_group == 3) the dy-th third of the tile's stage
  const bool grouped = MODE3 && p.a_group == 3;
  const uint32_t dy16 = MODE3 ? (grouped ? (uint32_t)p.a_stage_bytes / 48u : 0u) : (uint32_t)p.wp1 * row16;
  const int kcpt = p.kc_per_tap, a_stages = p.a_stages, b_stages = p.b_stages;
  const uint32_t bn = (uint32_t)p.bn;
  const bool skip_mma = (p.debug_flags & 2) != 0;     // timing experiment
  // this issuer's M halves: [h0, h1)
  const int h0 = p.n_issuers == 2 ? issuer : 0, h1 = p.n_issuers == 2 ? issuer + 1 : p.mh;
  const uint32_t half16 = (uint32_t)p.half_rows * row16;           // M halves: 128 rows apart (126 with fold)
  const int ndx = p.fold ? 1 : 3;                                   // fold: the filter columns live in N, one chain per filter row
  const uint32_t a_lo_base = desc_lo(a_base) + (uint32_t)h0 * half16;
  const uint32_t b_lo_base = desc_lo(b_base);
  int as = 0, bs = 0, it = 0;
  uint32_t aph = 0, bph = 0;
  if (BRES) {
    mbar_wait(smem_u32(bres_bar), 0);
    tc_fence_after();
  }
  // walk mode (MODE3 only): tile i of the run uses the ring stages of slabs i, i+1, i+2 and frees only the oldest
  const int nbuf_log2 = p.nbuf_log2, nbuf_mask = (1 << p.nbuf_log2) - 1;      // accumulator ring: 2 x 256 or 4 x 128 columns
  const uint32_t buf_cols = 512u >> p.nbuf_log2;
  const bool walk = MODE3 && p.walk;
  const int tile_begin = walk ? (int)blockIdx.x * p.tiles_per_cta : (int)blockIdx.x;
  const int tile_end = walk ? min(tile_begin + p.tiles_per_cta, num_tiles) : num_tiles;
  const int tile_step = walk ? 1 : (int)gridDim.x;
  for (int tile = tile_begin; tile < tile_end; tile += tile_step, ++it) {
    const int buf = it & nbuf_mask;
    mbar_wait(smem_u32(&tmem_empty_bar[buf]), ((it >> nbuf_log2) & 1) ^ 1);
    tc_fence_after();
    const uint32_t d_tmem = tmem_base + buf * buf_cols + (uint32_t)h0 * bn;
    for (int kc = 0; kc < kcpt; ++kc) {
      if (!MODE3) {
        mbar_wait(smem_u32(&a_full[as]), aph);
        tc_fence_after();
      }
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
        int sa = as;                 // ring stage of this filter row's slab
        if (MODE3 && (!grouped || dy == 0)) {
          uint32_t ph = aph;
          if (walk && dy > 0) {      // `as` moved on after filter row 0: rows 1, 2 sit in the next two stages
            sa = as + dy - 1;
            if (sa >= a_stages) { sa -= a_stages; ph ^= 1; }
          }
          // (walk: two of the three slabs were already waited for by the previous tile)
          if (!walk || dy == 2 || it == 0) {
            mbar_wait(smem_u32(&a_full[sa]), ph);
            tc_fence_after();
          }
        }
        const uint32_t a_row = a_lo_base + (uint32_t)sa * a_stage16 + (uint32_t)dy * dy16;
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          if (dx >= ndx) break;
          const int tap = dy * 3 + dx;
          uint32_t b_lo;
          if (BRES) {
            b_lo = b_lo_base + (uint32_t)((p.fold ? dy : tap) * kcpt + kc) * b16;
          } else {
            mbar_wait(smem_u32(&b_full[bs]), bph);
            tc_fence_after();
            b_lo = b_lo_base + (uint32_t)bs * b16;
          }
          const uint32_t a_lo = a_row + (uint32_t)dx * row16;
          for (int h = h0; h < h1 && !skip_mma; ++h) {
            const uint32_t ah = a_lo + (uint32_t)(h - h0) * half16;
#pragma unroll
            for (int k = 0; k < TC_BK / 16; ++k) {
              if (PAIR)
                tc_mma_f16_2sm(d_tmem + (uint32_t)(h - h0) * bn, desc_pack(ah + 2 * k), desc_pack(b_lo + 2 * k), idesc,
                               (tap == 0 && k == 0) ? (kc != 0 ? 1u : 0u) : 1u);
              else
                tc_mma_f16(d_tmem + (uint32_t)(h - h0) * bn, desc_pack(ah + 2 * k), desc_pack(b_lo + 2 * k), idesc,
                           (tap == 0 && k == 0) ? (kc != 0 ? 1u : 0u) : 1u);
            }
          }
          if (!BRES) {
            if (PAIR) tc_commit_2sm(smem_u32(&b_empty[bs]));
            else if (p.cluster == 2) tc_commit_mc(smem_u32(&b_empty[bs]), (uint16_t)3);      // frees the stage in both CTAs
            else tc_commit(smem_u32(&b_empty[bs]));
            if (++bs == b_stages) { bs = 0; bph ^= 1; }
          }
        }
        if (MODE3 && (grouped ? dy == 2 : (!walk || dy == 0))) {
          if (PAIR) tc_commit_2sm(smem_u32(&a_empty[as]));
          else tc_commit(smem_u32(&a_empty[as]));
          if (++as == a_stages) { as = 0; aph ^= 1; }
        }
      }
      if (!MODE3) {
        if (PAIR) tc_commit_2sm(smem_u32(&a_empty[as]));
        else tc_commit(smem_u32(&a_empty[as]));
        if (++as == a_stages) { as = 0; aph ^= 1; }
      }
    }
    if (PAIR) tc_commit_2sm(smem_u32(&tmem_full_bar[buf]));
    else tc_commit(smem_u32(&tmem_full_bar[buf]));
  }
}

// ------------------------------------------------------------------------------------------ slab-mode kernel
// 3x3 convolutions only.  For a tile of mh*128 consecutive PF rows and one block of 64 channels, the A rows of
// ALL nine taps come from one contiguous run of rows (slab_mode 1: mh*128 + 2*(w+1) + 2 rows) or from three runs,
// one per filter row (slab_mode 3: 3 x (mh*128 + 2) rows, used when the image is wide).  The slab is fetched
// once; each tap's A operand is a row-shifted view of it: shared-memory descriptor start = slab + off*128 B (the
// 128B swizzle is a function of the absolute shared-memory address, so TMA's layout and the MMA's view agree
// without touching the descriptor's base-offset field — verified against a reference convolution on B200).  Compared with one TMA tile per tap this
// cuts the L2 -> SMEM traffic of A by 9x/(1.2 ... 3x), which is what bounds the 64/128-channel 224^2/112^2 layers.
// B tiles stream through their own ring (kc-major, tap-minor) or, when the whole layer's B fits (<= 80 KB),
// stay resident for the lifetime of the persistent CTA.  With mh == 2 every B tile feeds two 128-row MMAs.
constexpr int TC_A_MAX_STAGES = 6;
#ifndef LRPX_TC_PAIR_DEFAULT
#define LRPX_TC_PAIR_DEFAULT true
#endif

// PAIR is a template parameter, not p.pair: a kernel that CONTAINS cta_group::2 instructions can only be launched as a
// cluster of CTA pairs (a plain launch of it fails with cudaErrorInvalidClusterSize, measured), so the pair-mode code lives
// in its own instantiations.
template <int EPI, bool PAIR = false>
__global__ void __launch_bounds__(TC_THREADS, 1)
tc_conv_slab_kernel(const __grid_constant__ CUtensorMap tmA0, const __grid_constant__ CUtensorMap tmA1,
                    const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmBh,
                    const __grid_constant__ CUtensorMap tmO, const TcParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  __shared__ __align__(8) uint64_t a_full[TC_A_MAX_STAGES];
  __shared__ __align__(8) uint64_t a_empty[TC_A_MAX_STAGES];
  __shared__ __align__(8) uint64_t b_full[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t b_empty[TC_MAX_STAGES];
  __shared__ __align__(8) uint64_t bres_bar;
  __shared__ __align__(8) uint64_t tmem_full_bar[4];
  __shared__ __align__(8) uint64_t tmem_empty_bar[4];
  __shared__ uint32_t tmem_base_slot;
  // EPI_INPUT3: [accumulator buffer][tile parity of the warp set][M half][quarter][2][8].  A warp writes its boundary
  // rows BEFORE the named barrier of a tile and reads its neighbours' right after it; with two copies alternating per
  // tile a slot is rewritten only after the barrier of the tile in between, which every reader of the old value has
  // passed its reads to reach.
  __shared__ float in3_scratch[2][4][128];      // INPUT3: [buffer][tile parity][2 halves x 64]; MUL_FOLD: [buffer][unit][4 quarters x 2 x 16]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  const uint32_t b_bytes = (uint32_t)p.bn * TC_BK * 2;
  const uint32_t a_base = smem_base;
  const uint32_t b_base = smem_base + (uint32_t)p.a_stages * p.a_stage_bytes;
  const int num_tiles = p.tiles_sched;
  const int tile_rows = p.tile_stride;         // row distance of the M tiles (= output rows per tile; walk: one image row);
                                               // with fold the computed rows start one row earlier
  // Row walk (p.walk; the 224^2 first layer): CTA c takes tiles [c * tiles_per_cta, ...) one image row (w + 1 PF rows)
  // apart.  Slab j of tile m starts at row (m + j - 1)(w + 1) - 1 = slab j - 1 of tile m + 1: after the first tile of a run
  // only ONE new slab is fetched per tile (L2 -> SM traffic of A 258/225 = 1.15x the rows instead of 3 x 258/252 = 3.07x,
  // which is what bound the layer).  A tile still computes 252 rows; the rows past the stride are the next tile's.
  const int tile_begin = p.walk ? (int)blockIdx.x * p.tiles_per_cta : (int)blockIdx.x;
  const int tile_end = p.walk ? min(tile_begin + p.tiles_per_cta, num_tiles) : num_tiles;
  const int tile_step = p.walk ? 1 : (int)gridDim.x;
  const int n_slabs = p.slab_mode == 1 ? 1 : 3;

  if (threadIdx.x == 0) {
    // "empty" / "accumulator ready" barriers collect one tcgen05.commit per issuer warp
    for (int s = 0; s < p.a_stages; ++s) {
      mbar_init(smem_u32(&a_full[s]), 1);
      mbar_init(smem_u32(&a_empty[s]), p.n_issuers);
    }
    for (int s = 0; s < p.b_stages; ++s) {
      mbar_init(smem_u32(&b_full[s]), 1);
      // cluster (multicast B): both CTAs' issuers release a B stage; pair: only the leader's issuers commit (to both CTAs)
      mbar_init(smem_u32(&b_empty[s]), PAIR ? p.n_issuers : p.n_issuers * p.cluster);
    }
    mbar_init(smem_u32(&bres_bar), 1);
    for (int b = 0; b < 4; ++b) {
      mbar_init(smem_u32(&tmem_full_bar[b]), p.n_issuers);
      // pair: the leader's issuers wait for the epilogue warps of BOTH CTAs (the peer's arrive remotely)
      // (first-layer epilogues: only the 4 * mh warps of the tile's set read the buffer, see the epilogue loop)
      mbar_init(smem_u32(&tmem_empty_bar[b]), (EPI == LRPX_TC_EPI_INPUT || is_input3(EPI))
                                                  ? 4 * p.mh : (PAIR ? 2 * TC_EPI_WARPS : TC_EPI_WARPS));
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
  }
  if (PAIR) cluster_sync_all();               // both CTAs are resident before the paired TMEM allocation
  if (warp == 1) {
    if (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_slot)),
                   "r"(512u)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  if (p.cluster == 2) cluster_sync_all();      // the peer's barriers exist before any multicast traffic or remote arrive
  const uint32_t tmem_base = tmem_base_slot;
  const uint32_t pair_rank = PAIR ? cluster_ctarank() : 0u;

  if (warp == 0) {
    // ================================ A producer (one thread)
    if (elect_one()) {
      int as = 0;
      uint32_t aph = 0;
      const uint32_t a_tx = (uint32_t)p.slab_rows * (TC_BK * 2);
      for (int tile = tile_begin; tile < tile_end; tile += tile_step) {
        int m_tile, n_tile_unused;
        tile_coords(p, tile, m_tile, n_tile_unused);
        const int m0 = m_tile * tile_rows;             // fold: P' rows start at m0 - 1, which is where the slabs start anyway
        const int j0 = (p.walk && tile != tile_begin) ? n_slabs - 1 : 0;      // walk: slabs 0, 1 are the previous tile's 1, 2
        for (int kc = 0; kc < p.kc_per_tap; ++kc) {
          if (p.a_group == 3) {                        // one ring stage for the tile's three slabs (not with PAIR / walk)
            mbar_wait_ns(smem_u32(&a_empty[as]), aph ^ 1, (uint32_t)p.sleep_ns);
            const uint32_t fb = smem_u32(&a_full[as]);
            const uint32_t dst = a_base + (uint32_t)as * p.a_stage_bytes;
            const int kca = (p.a_wrap && kc >= p.a_wrap) ? kc - p.a_wrap : kc;
            if (p.debug_flags & 4) {
              mbar_arrive(fb);
            } else {
              mbar_expect_tx(fb, 3 * a_tx);
              for (int j = 0; j < 3; ++j) {
                const int row0 = m0 + (j - 1) * p.wp1 - 1;
                const uint32_t dj = dst + (uint32_t)j * ((uint32_t)p.a_stage_bytes / 3u);
                tma_load_2d(dj, &tmA0, fb, kca * TC_BK, row0);
                if (p.box1_rows) tma_load_2d(dj + (uint32_t)p.box0_rows * (TC_BK * 2), &tmA1, fb, kca * TC_BK, row0 + p.box0_rows);
              }
            }
            if (++as == p.a_stages) { as = 0; aph ^= 1; }
            continue;
          }
          for (int j = j0; j < n_slabs; ++j) {         // one ring stage per slab
            mbar_wait_ns(smem_u32(&a_empty[as]), aph ^ 1, (uint32_t)p.sleep_ns);
            const uint32_t fb = smem_u32(&a_full[as]);
            const uint32_t dst = a_base + (uint32_t)as * p.a_stage_bytes;
            if (p.debug_flags & 4) {          // timing experiment: no A traffic
              mbar_arrive(fb);
            } else if (PAIR) {
              // each CTA fetches its own slab into its own shared memory; both signal the LEADER's barrier, on which
              // the leader expects the bytes of both
              const uint32_t fbl = pair_rank ? mapa_u32(fb, 0) : fb;
              if (!pair_rank) mbar_expect_tx(fb, 2 * a_tx);
              const int row0 = (p.slab_mode == 1) ? m0 - p.wp1 - 1 : m0 + (j - 1) * p.wp1 - 1;
              const int kca = (p.a_wrap && kc >= p.a_wrap) ? kc - p.a_wrap : kc;
              tma_load_2d_2sm(dst, &tmA0, fbl, kca * TC_BK, row0);
              if (p.box1_rows) tma_load_2d_2sm(dst + (uint32_t)p.box0_rows * (TC_BK * 2), &tmA1, fbl, kca * TC_BK, row0 + p.box0_rows);
            } else {
              mbar_expect_tx(fb, a_tx);
              const int row0 = (p.slab_mode == 1) ? m0 - p.wp1 - 1 : m0 + (j - 1) * p.wp1 - 1;
              const int kca = (p.a_wrap && kc >= p.a_wrap) ? kc - p.a_wrap : kc;    // hi | lo | hi view of a split row
              tma_load_2d(dst, &tmA0, fb, kca * TC_BK, row0);
              if (p.box1_rows) tma_load_2d(dst + (uint32_t)p.box0_rows * (TC_BK * 2), &tmA1, fb, kca * TC_BK, row0 + p.box0_rows);
            }
            if (++as == p.a_stages) { as = 0; aph ^= 1; }
          }
        }
      }
    }
  } else if (warp == TC_BPROD_WARP) {
    // ================================ B producer (one thread)
    if (elect_one()) {
      if (p.b_resident && PAIR) {
        // pair: this CTA keeps rows [rank*bn/2, +bn/2) of every B tile (half-size pitch); the leader's barrier counts both
        const uint32_t bb = smem_u32(&bres_bar);
        const uint32_t bbl = pair_rank ? mapa_u32(bb, 0) : bb;
        const uint32_t hb = b_bytes >> 1;
        if (!pair_rank) mbar_expect_tx(bb, (uint32_t)(p.taps * p.kc_per_tap) * b_bytes);
        for (int tap = 0; tap < p.taps; ++tap)
          for (int kc = 0; kc < p.kc_per_tap; ++kc)
            tma_load_2d_2sm(b_base + (uint32_t)(tap * p.kc_per_tap + kc) * hb, &tmBh, bbl, tap * p.cin + kc * TC_BK,
                            (int)pair_rank * (p.bn >> 1));
      } else if (p.b_resident) {
        const uint32_t bb = smem_u32(&bres_bar);
        mbar_expect_tx(bb, (uint32_t)(p.taps * p.kc_per_tap) * b_bytes);
        for (int tap = 0; tap < p.taps; ++tap)
          for (int kc = 0; kc < p.kc_per_tap; ++kc)
            tma_load_2d(b_base + (uint32_t)(tap * p.kc_per_tap + kc) * b_bytes, &tmB, bb, tap * p.cin + kc * TC_BK, 0);
      } else if (PAIR) {
        int bs = 0;
        uint32_t bph = 0;
        const uint32_t hb = b_bytes >> 1;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
          int m_tile_unused, n_tile;
          tile_coords(p, tile, m_tile_unused, n_tile);
          const int n0 = n_tile * p.bn;
          for (int kc = 0; kc < p.kc_per_tap; ++kc)
            for (int tap = 0; tap < p.taps; ++tap) {
              mbar_wait_ns(smem_u32(&b_empty[bs]), bph ^ 1, (uint32_t)p.sleep_ns);
              const uint32_t bb = smem_u32(&b_full[bs]);
              const uint32_t bbl = pair_rank ? mapa_u32(bb, 0) : bb;
              if (!pair_rank) mbar_expect_tx(bb, b_bytes);
              tma_load_2d_2sm(b_base + (uint32_t)bs * hb, &tmBh, bbl, tap * p.cin + kc * TC_BK, n0 + (int)pair_rank * (p.bn >> 1));
              if (++bs == p.b_stages) { bs = 0; bph ^= 1; }
            }
        }
      } else {
        int bs = 0;
        uint32_t bph = 0;
        // cluster mode: this CTA fetches HALF of every B tile (rows [rank*bn/2, +bn/2)) and multicasts it into both
        // CTAs of the pair; a stage is free once the issuers of BOTH CTAs have committed it (b_empty counts them all)
        const uint32_t rank = p.cluster == 2 ? cluster_ctarank() : 0u;
        const uint32_t half_bytes = b_bytes >> 1;
        for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
          int m_tile_unused, n_tile;
          tile_coords(p, tile, m_tile_unused, n_tile);
          const int n0 = n_tile * p.bn;
          for (int kc = 0; kc < p.kc_per_tap; ++kc)
            for (int tap = 0; tap < p.taps; ++tap) {
              mbar_wait_ns(smem_u32(&b_empty[bs]), bph ^ 1, (uint32_t)p.sleep_ns);
              const uint32_t bb = smem_u32(&b_full[bs]);
              mbar_expect_tx(bb, b_bytes);
              if (p.cluster == 2)
                tma_load_2d_mc(b_base + (uint32_t)bs * b_bytes + rank * half_bytes, &tmBh, bb, tap * p.cin + kc * TC_BK,
                               n0 + (int)rank * (p.bn >> 1), (uint16_t)3);
              else
                tma_load_2d(b_base + (uint32_t)bs * b_bytes, &tmB, bb, tap * p.cin + kc * TC_BK, n0);
              if (++bs == p.b_stages) { bs = 0; bph ^= 1; }
            }
        }
      }
    }
  } else if (warp == 1 || warp == TC_MMA2_WARP) {
    // ================================ MMA issuers (one elected thread per issuer warp)
    const int issuer = warp == 1 ? 0 : 1;
    // pair mode: only the leader CTA issues (its MMAs run on both SMs)
    if (issuer < p.n_issuers && pair_rank == 0 && elect_one()) {
#define LRPX_SLAB_LOOP(BRES, MODE3, PAIR)                                                                             \
  do {                                                                                                                \
    if (issuer == 0)                                                                                                  \
      slab_mma_loop<BRES, MODE3, 0, PAIR>(p, a_full, a_empty, b_full, b_empty, &bres_bar, tmem_full_bar,              \
                                          tmem_empty_bar, a_base, b_base, tmem_base, num_tiles);                      \
    else                                                                                                              \
      slab_mma_loop<BRES, MODE3, 1, PAIR>(p, a_full, a_empty, b_full, b_empty, &bres_bar, tmem_full_bar,              \
                                          tmem_empty_bar, a_base, b_base, tmem_base, num_tiles);                      \
  } while (0)
      if (PAIR) {
        if (p.b_resident) {
          if (p.slab_mode == 3) LRPX_SLAB_LOOP(true, true, PAIR); else LRPX_SLAB_LOOP(true, false, PAIR);
        } else {
          if (p.slab_mode == 3) LRPX_SLAB_LOOP(false, true, PAIR); else LRPX_SLAB_LOOP(false, false, PAIR);
        }
      } else if (p.b_resident) {
        if (p.slab_mode == 3) LRPX_SLAB_LOOP(true, true, false); else LRPX_SLAB_LOOP(true, false, false);
      } else {
        if (p.slab_mode == 3) LRPX_SLAB_LOOP(false, true, false); else LRPX_SLAB_LOOP(false, false, false);
      }
#undef LRPX_SLAB_LOOP
    }
    __syncwarp();
  } else if (warp >= 2 && warp < 2 + TC_EPI_WARPS) {
    // ================================ epilogue warps
    const int quarter = warp & 3;
    // First-layer epilogues (one unit per M half): the warps form two sets that take alternate tiles (run_epilogue_tile).  A
    // warp walks ONLY its own set's tiles — a tile of that layer costs the SM ~5300 warp instructions, it is bound by
    // instruction issue, and a third of them were the other set's (and the unit-less warps') trips through this loop just to
    // hand the buffer back; the buffer's "empty" barrier counts the 4 * mh warps that actually read it.
    constexpr bool kSets = EPI == LRPX_TC_EPI_INPUT || is_input3(EPI);
    const int sub0 = (warp - 2) >> 2;
    int it = 0, it_step = 1;
    bool idle = false;
    if (kSets) {
      if ((sub0 & 1) >= p.mh) idle = true;       // no unit for this warp (mh == 1)
      else { it = sub0 >> 1; it_step = 2; }
    }
    for (int tile = tile_begin + it * tile_step; !idle && tile < tile_end; tile += it_step * tile_step, it += it_step) {
      // accumulator ring: two buffers of 256 TMEM columns, or four of 128 when a tile's accumulators fit (mh * bn <= 128):
      // the MMAs then run up to four tiles ahead of the epilogue, which is what a layer whose tile time is the round trip
      // commit -> epilogue wake-up -> TMEM read -> release -> issuer wake-up needs (the first layer: 24 columns per half)
      const int buf = it & ((1 << p.nbuf_log2) - 1);
      const uint32_t acc_phase = (it >> p.nbuf_log2) & 1;
      int m_tile, n_tile;
      tile_coords(p, tile, m_tile, n_tile);
      if (!is_input3(EPI)) {                    // INPUT3 waits inside its epilogue, after its loads are in flight
        mbar_wait_ns(smem_u32(&tmem_full_bar[buf]), acc_phase, (uint32_t)p.sleep_ns);
        tc_fence_after();
      }
      const int tile_pf = tile + 2 * tile_step;           // L2 prefetch distance: two of this CTA's tiles ahead
      int m_pf = 0, n_pf = -1;
      if (tile_pf < tile_end) tile_coords(p, tile_pf, m_pf, n_pf);
      const int pf_row = (n_pf == n_tile) ? m_pf * tile_rows + quarter * 32 + lane : -1;
      const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * (512u >> p.nbuf_log2);
      const uint32_t stage = (EPI == LRPX_TC_EPI_MUL && p.store_off) ? smem_base + (uint32_t)p.store_off + (uint32_t)(warp - 2) * 1024u : 0u;
      uint32_t rel_bar = smem_u32(&tmem_empty_bar[buf]);
      if (PAIR) rel_bar = mapa_u32(rel_bar, 0);          // shared::cluster address of the LEADER's barrier (both ranks)
      run_epilogue_tile<EPI>(p, m_tile * tile_rows - p.fold + quarter * 32 + lane, taddr, n_tile, (warp - 2) >> 2, p.mh,
                             pf_row, rel_bar, stage, &tmO,
                             is_input3(EPI) ? &in3_scratch[it & 1][(it >> 1) & 1][0]
                                            : (EPI == TC_EPI_MUL_FOLD ? &in3_scratch[it & 1][0][0] : nullptr),
                             quarter, it, smem_u32(&tmem_full_bar[buf]), acc_phase);
    }
    if (EPI == LRPX_TC_EPI_MUL && p.store_off) {      // the staging block must outlive the last tile store's read
      if (lane == 0) bulk_wait_read0();
      __syncwarp();
    }
  }

  tc_fence_before();
  __syncthreads();
  if (p.cluster == 2) cluster_sync_all();      // no CTA leaves while its peer may still multicast into it / arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    if (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
  }
}

// ------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  });
  return fn;
}

// 2-D bf16 tensor (rows x cols, cols contiguous), box = (64 cols, box_rows), SWIZZLE_128B, zero OOB fill
static int make_map_2d(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return LRPX_E_CUDA;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)TC_BK, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) rows=%llu cols=%llu box_rows=%u", (int)r, (unsigned long long)rows,
              (unsigned long long)cols, box_rows);
    return LRPX_E_CUDA;
  }
  return LRPX_OK;
}

// output tensor of the MUL epilogue: 2-D bf16 (rows x cols), box = (16 cols, 32 rows), SWIZZLE_32B
static int make_map_out(CUtensorMap* map, const void* base, uint64_t rows, uint64_t cols) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available");
    return LRPX_E_CUDA;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 2};
  cuuint32_t box[2] = {16, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_32B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled (output) failed (%d) rows=%llu cols=%llu", (int)r, (unsigned long long)rows,
              (unsigned long long)cols);
    return LRPX_E_CUDA;
  }
  return LRPX_OK;
}

template <int EPI>
static int launch_tc(const CUtensorMap& ma, const CUtensorMap& mb, const TcParams& p, int grid, cudaStream_t st) {
  static std::atomic<uint64_t> attr_done;
  const int rc = ensure_smem_attr(tc_conv_kernel<EPI>, TC_SMEM_BYTES, attr_done);
  if (rc != LRPX_OK) return rc;
  tc_conv_kernel<EPI><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(ma, mb, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("tc_conv_kernel launch failed: %s", cudaGetErrorString(e));
    return LRPX_E_CUDA;
  }
  return LRPX_OK;
}

template <int EPI, bool PAIR>
static int launch_tc_slab_impl(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mb, const CUtensorMap& mbh,
                               const CUtensorMap& mo, const TcParams& p, int grid, cudaStream_t st);

template <int EPI>
static int launch_tc_slab(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mb, const CUtensorMap& mbh,
                          const CUtensorMap& mo, const TcParams& p, int grid, cudaStream_t st) {
  if constexpr (EPI == LRPX_TC_EPI_MUL || EPI == LRPX_TC_EPI_MUL_UNPOOL || EPI == LRPX_TC_EPI_MULX ||
                EPI == LRPX_TC_EPI_MULX_UNPOOL || EPI == TC_EPI_MULX_S || EPI == TC_EPI_MULX_UNPOOL_S) {
    if (p.pair) return launch_tc_slab_impl<EPI, true>(ma0, ma1, mb, mbh, mo, p, grid, st);
  }
  if (p.pair) {
    set_error("pair mode is not built for this epilogue");
    return LRPX_E_INVALID;
  }
  return launch_tc_slab_impl<EPI, false>(ma0, ma1, mb, mbh, mo, p, grid, st);
}

template <int EPI, bool PAIR>
static int launch_tc_slab_impl(const CUtensorMap& ma0, const CUtensorMap& ma1, const CUtensorMap& mb, const CUtensorMap& mbh,
                               const CUtensorMap& mo, const TcParams& p, int grid, cudaStream_t st) {
  static std::atomic<uint64_t> attr_done;
  const int rc = ensure_smem_attr(tc_conv_slab_kernel<EPI, PAIR>, TC_SMEM_BYTES, attr_done);
  if (rc != LRPX_OK) return rc;
  if (p.cluster == 2) {
    // GPCs with an odd number of SMs cannot host a pair on their last SM: a persistent grid must not exceed the
    // number of clusters that are co-resident, or the left-over pair would run after everyone else
    static int max_clusters = -1;
    if (max_clusters < 0) {
      cudaLaunchConfig_t q{};
      q.gridDim = dim3(2 * 148);
      q.blockDim = dim3(TC_THREADS);
      q.dynamicSmemBytes = TC_SMEM_BYTES;
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = 2; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      q.attrs = qa; q.numAttrs = 1;
      int n = 0;
      if (cudaOccupancyMaxActiveClusters(&n, tc_conv_slab_kernel<EPI, PAIR>, &q) != cudaSuccess || n <= 0) n = 64;
      max_clusters = n;
    }
    if (grid > 2 * max_clusters) grid = 2 * max_clusters;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)grid);
    cfg.blockDim = dim3(TC_THREADS);
    cfg.dynamicSmemBytes = TC_SMEM_BYTES;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    cudaError_t le = cudaLaunchKernelEx(&cfg, tc_conv_slab_kernel<EPI, PAIR>, ma0, ma1, mb, mbh, mo, p);
    if (le != cudaSuccess) {
      set_error("tc_conv_slab_kernel cluster launch failed: %s", cudaGetErrorString(le));
      return LRPX_E_CUDA;
    }
    return LRPX_OK;
  }
  tc_conv_slab_kernel<EPI, PAIR><<<grid, TC_THREADS, TC_SMEM_BYTES, st>>>(ma0, ma1, mb, mbh, mo, p);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("tc_conv_slab_kernel launch failed: %s", cudaGetErrorString(e));
    return LRPX_E_CUDA;
  }
  return LRPX_OK;
}

// Picks the slab-mode configuration (see tc_conv_slab_kernel).  Returns false when nothing fits.
//   mh = 2 (256-row tiles, one issuer warp per half) whenever two accumulators of the tile fit one TMEM buffer
//   (bn <= 128); slab_mode 1 when the single slab is the smaller fetch and fits two TMA boxes, else one slab per
//   filter row; B resident when the whole layer's B fits next to >= 2 (mode 1) / 4 (mode 3) A stages.
static bool plan_slab(TcParams& p, int reserve, bool pair) {
  const int budget = TC_SMEM_BYTES - 1024 - reserve;
  const int b_bytes = p.bn * TC_BK * 2;
  // pair mode: each CTA of the pair keeps half of every B tile, so a layer's B is resident from twice the size on
  const long long b_total = (long long)p.taps * p.kc_per_tap * b_bytes / (pair ? 2 : 1);
  const char* env_mh = getenv("LRPX_TC_MH");             // experiment switches (timing probes only)
  const char* env_iss = getenv("LRPX_TC_ISSUERS");
  const char* env_res = getenv("LRPX_TC_RES3");           // "0": do not trade slab mode 1 for a resident B
  const int mh_max = (env_mh && env_mh[0] == '1') ? 1 : 2;
  auto commit = [&](int mode, int mh, int slab_rows, int slab_bytes, int a_stages, int b_stages, bool res) {
    p.slab_mode = mode; p.mh = mh; p.slab_rows = slab_rows;
    p.n_issuers = (mh == 2 && !(env_iss && env_iss[0] == '1')) ? 2 : 1;
    p.box0_rows = slab_rows < 256 ? slab_rows : 256;
    p.box1_rows = slab_rows - p.box0_rows;
    p.a_stage_bytes = slab_bytes;
    p.a_stages = a_stages; p.b_stages = b_stages; p.b_resident = res ? 1 : 0;
    return true;
  };
  for (int mh = p.bn <= 128 ? mh_max : 1; mh >= 1; --mh) {
    const int rows1 = mh * TC_BM + 2 + 2 * p.wp1, rows3 = mh * TC_BM + 2;
    const int bytes1 = ((rows1 * TC_BK * 2) + 1023) & ~1023, bytes3 = ((rows3 * TC_BK * 2) + 1023) & ~1023;
    const bool mode1_ok = rows1 <= 3 * rows3 && rows1 <= 512;
    // (1) resident B: streaming B costs more shared-memory ingest (and one barrier round trip per tap) than the
    //     A slabs do, so it is worth fewer A stages and even the larger per-filter-row slabs of mode 3
    if (p.num_n_tiles == 1) {
      if (mode1_ok)
        for (int a_stages = 3; a_stages >= 2; --a_stages)
          if ((long long)a_stages * bytes1 + b_total <= budget) return commit(1, mh, rows1, bytes1, a_stages, 0, true);
      if (!mode1_ok || !(env_res && env_res[0] == '0'))
        for (int a_stages = TC_A_MAX_STAGES; a_stages >= 2; --a_stages)
          if ((long long)a_stages * bytes3 + b_total <= budget) return commit(3, mh, rows3, bytes3, a_stages, 0, true);
    }
    // (2) B streamed through its own ring
    const int mode = mode1_ok ? 1 : 3;
    const int slab_rows = mode == 1 ? rows1 : rows3, slab_bytes = mode == 1 ? bytes1 : bytes3;
    const int min_a = mode == 1 ? 2 : 4, max_a = mode == 1 ? 3 : TC_A_MAX_STAGES;
    for (int a_stages = max_a; a_stages >= min_a; --a_stages) {
      const int left = budget - a_stages * slab_bytes;
      int b_stages = left / b_bytes;
      if (b_stages > TC_MAX_STAGES) b_stages = TC_MAX_STAGES;
      // the B ring has to cover the TMA latency: >= 4 tiles and >= 48 KB in flight unless A is at its minimum
      if (b_stages < 3) continue;
      if (a_stages > min_a && (b_stages < 4 || b_stages * b_bytes < 48 * 1024)) continue;
      return commit(mode, mh, slab_rows, slab_bytes, a_stages, b_stages, false);
    }
  }
  return false;
}

static int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

}  // namespace lrpx

using namespace lrpx;

extern "C" int lrpx_tc_conv(const lrpx_tc_conv_args* a, void* stream) {
  LRPX_CHECK_ARG(a, "null args");
  LRPX_CHECK_ARG(a->n_img > 0 && a->h >= 0 && a->w >= 0, "bad image dimensions");
  LRPX_CHECK_ARG(a->cin > 0 && a->cin % TC_BK == 0, "cin must be a multiple of 64");
  LRPX_CHECK_ARG(a->ksize == 1 || a->ksize == 3, "ksize must be 1 or 3");
  LRPX_CHECK_ARG(a->a && a->wt && a->out, "null pointer");
  LRPX_CHECK_ARG(a->ncol > 0 && (a->ncol % 16 == 0 || (a->epilogue == LRPX_TC_EPI_INPUT3 && a->ncol == 24)),
                 "ncol must be a multiple of 16");
  const int epi = a->epilogue;
  TcParams p{};
  p.h = a->h; p.w = a->w; p.wp1 = a->w + 1;
  p.blk = (a->h + 1) * (a->w + 1);
  {
    auto magic = [](int d, uint32_t& mul, int& sh) {      // n / d == (n * mul) >> sh for 0 <= n < 2^31
      int s = 0;
      while ((1LL << s) < d) ++s;
      sh = 31 + s;
      mul = (uint32_t)((((unsigned long long)1 << sh) + (unsigned long long)d - 1) / (unsigned long long)d);
    };
    magic(p.blk, p.blk_mul, p.blk_sh);
    magic(p.wp1, p.wp1_mul, p.wp1_sh);
  }
  long long m_total = (long long)a->n_img * p.blk;
  LRPX_CHECK_ARG(m_total < (1LL << 31) - 4096, "too many pixel rows for one call");
  p.m_total = (int)m_total;
  p.cin = a->cin; p.ncol = a->ncol;
  p.taps = a->ksize * a->ksize;
  p.kc_per_tap = a->cin / TC_BK;
  p.bias = a->bias; p.gain = reinterpret_cast<const __nv_bfloat16*>(a->gain);
  p.row_img = a->row_img; p.pool_idx = a->pool_idx; p.x = a->x; p.x1 = a->x1; p.out = a->out; p.out2 = a->out2;
  p.gain_mode = a->gain_mode;
  // ---- general modes
  const int a_phys = a->a_phys > 0 ? a->a_phys : a->cin;
  LRPX_CHECK_ARG(a_phys % TC_BK == 0 && a_phys <= a->cin && (a_phys == a->cin || a->cin <= 2 * a_phys),
                 "a_phys must be a multiple of 64 with cin/2 <= a_phys <= cin");
  p.a_wrap = a_phys < a->cin ? a_phys / TC_BK : 0;
  p.groups = a->groups > 0 ? a->groups : 1;
  p.split = a->split; p.n_acc = a->n_acc; p.rule = a->rule; p.zbias = a->zbias;
  p.alpha = a->alpha; p.beta = a->beta; p.gain2 = a->gain2; p.out3 = a->out3;
  p.add = a->add; p.add_pitch = a->add_pitch; p.gain3 = a->gain3; p.gain4 = a->gain4;
  p.bn_w = a->bn_w; p.bn_b = a->bn_b; p.idn = a->idn; p.hd = a->hd; p.out4 = a->out4; p.out5 = a->out5;
  p.fwd_flags = a->fwd_flags;
  LRPX_CHECK_ARG(!a->cam_rows || (epi == LRPX_TC_EPI_INPUT3 && a->rule == 3),
                 "cam_rows: Guided Grad-CAM's factor needs the INPUT3 epilogue and the guided rule (3)");
  LRPX_CHECK_ARG(!a->cam_rows || (a->cam_kw && a->cam_w > 0 && a->cam_w <= 64), "cam_rows needs cam_kw and 0 < cam_w <= 64");
  p.cam_rows = a->cam_rows; p.cam_kw = a->cam_kw; p.cam_w = a->cam_w;

  if (epi == LRPX_TC_EPI_FWDX) {
    LRPX_CHECK_ARG(a->out2 && a->n_acc >= 1 && a->n_acc <= 3 && a->ncol % a->n_acc == 0, "FWDX: out2 and n_acc in 1..3");
    LRPX_CHECK_ARG((a->rule == 0 && a->n_acc >= 2) || (a->rule >= 1 && a->rule <= 3 && a->n_acc == 1),
                   "FWDX: alpha-beta needs W and W+ (n_acc >= 2); epsilon / gradient / guided n_acc == 1");
    LRPX_CHECK_ARG(a->out3 == nullptr || a->n_acc == 3 || a->idn, "FWDX: out3 needs n_acc == 3 (neg-net gain) or idn (identity-branch gain)");
    LRPX_CHECK_ARG((a->bn_w == nullptr) == (a->bn_b == nullptr), "FWDX: bn_w and bn_b go together");
    LRPX_CHECK_ARG(!(a->fwd_flags & 2) || (a->h % 2 == 0 && a->w % 2 == 0 && !a->idn && !a->hd), "FWDX: strided store needs even h, w and no idn / hd");
    const int cout = a->ncol / a->n_acc;
    LRPX_CHECK_ARG(cout % 32 == 0, "FWDX: output channels must be a multiple of 32");
    const int cap = a->n_acc == 3 ? 64 : (a->n_acc == 2 ? 128 : 256);      // n_acc * half <= 256 TMEM columns per buffer
    p.half = cout < cap ? cout : cap;
    LRPX_CHECK_ARG(cout % p.half == 0, "FWDX: output channels must divide into tiles of 64 / 128 / 256");
    p.bn = a->n_acc * p.half;
    p.cout = cout;
    p.out_c = cout;
    const char* env_fs = getenv("LRPX_TC_FWD_SIMPLE");       // "0": always the general epilogue (A/B runs)
    p.fwd_simple = (a->n_acc <= 2 && !a->bn_w && !a->idn && !a->hd && !a->out3 && !a->out4 && !a->out5 && a->fwd_flags == 0 &&
                    !(env_fs && env_fs[0] == '0')) ? 1 : 0;
  } else if (epi == LRPX_TC_EPI_MULX || epi == LRPX_TC_EPI_MULX_UNPOOL) {
    LRPX_CHECK_ARG(a->gain && (p.groups == 1 || (p.groups == 2 && a->gain2)), "MULX: gain (and gain2 for two groups) required");
    LRPX_CHECK_ARG(a->ncol % 32 == 0, "ncol must be a multiple of 32 for this epilogue");
    LRPX_CHECK_ARG(!a->add || (epi == LRPX_TC_EPI_MULX && a->add_pitch >= a->ncol),
                   "MULX add: add_pitch >= ncol required; not with UNPOOL");
    LRPX_CHECK_ARG(!(a->out2 && p.groups == 2) || !p.split, "MULX: separate group tensors (out2) are bf16 only");
    p.bn = a->ncol <= 256 ? a->ncol : 256;
    LRPX_CHECK_ARG(a->ncol % p.bn == 0, "ncol must be <= 256 or a multiple of 256");
    {
      const char* env_ms = getenv("LRPX_TC_MULX_SIMPLE");    // "0": always the general epilogue (A/B runs)
      p.mulx_simple = (p.groups == 1 && !a->add && !a->out2 && !(env_ms && env_ms[0] == '0')) ? 1 : 0;
    }
    p.out_c = (a->out2 && p.groups == 2) ? a->ncol : a->ncol * p.groups * (p.split ? 2 : 1);
  } else if (epi == LRPX_TC_EPI_FWD_GAIN) {
    // Wt holds, per tile of `half` output channels, the W rows followed by the W+ rows: ncol = 2 * cout
    LRPX_CHECK_ARG(a->out2, "FWD_GAIN needs out2 (gain)");
    int cout = a->ncol / 2;
    LRPX_CHECK_ARG(cout % 32 == 0, "FWD_GAIN: output channels must be a multiple of 32");
    p.half = cout < 128 ? cout : 128;
    LRPX_CHECK_ARG(cout % p.half == 0, "FWD_GAIN: output channels must be <128 or a multiple of 128");
    p.bn = 2 * p.half;
    p.out_c = cout;
  } else if (epi == LRPX_TC_EPI_INPUT3) {
    LRPX_CHECK_ARG(a->ncol == 24 && a->x && a->ksize == 3, "INPUT3 epilogue: ncol must be 24, x set, 3x3");
    p.bn = 24;
    p.out_c = 3;
    p.taps = 3;           // B tiles per channel block: one per filter row (the filter columns live in N)
    p.fold = 1;
  } else if (epi == LRPX_TC_EPI_INPUT) {
    LRPX_CHECK_ARG(a->ncol == 16 && a->x, "INPUT epilogue: ncol must be 16 (3 W+ cols, 3 W- cols, padding) and x set");
    p.bn = 16;
    p.out_c = 3;
  } else {
    LRPX_CHECK_ARG(epi == LRPX_TC_EPI_MUL || epi == LRPX_TC_EPI_MUL_UNPOOL || epi == LRPX_TC_EPI_STORE_F32 ||
                       epi == LRPX_TC_EPI_FEAT || epi == LRPX_TC_EPI_FEAT_DIV,
                   "unknown epilogue");
    LRPX_CHECK_ARG(a->ncol % 32 == 0, "ncol must be a multiple of 32 for this epilogue");
    if (epi == LRPX_TC_EPI_FEAT || epi == LRPX_TC_EPI_FEAT_DIV) {
      LRPX_CHECK_ARG(a->x && a->ksize == 1, "FEAT epilogues: x required, ksize 1");
      LRPX_CHECK_ARG(epi == LRPX_TC_EPI_FEAT || a->x1, "FEAT_DIV needs x1");
    } else if (epi != LRPX_TC_EPI_STORE_F32) LRPX_CHECK_ARG(a->gain, "gain required");
    if (epi == LRPX_TC_EPI_MUL_UNPOOL) LRPX_CHECK_ARG(a->pool_idx, "pool_idx required");
    p.bn = a->ncol <= 256 ? a->ncol : 256;
    if (a->fwd_flags & LRPX_TC_FOLD_COLUMNS) {
      // Wt holds 3 * ncol rows (row dx * ncol + n, K ordered (filter row, channel)): see epi_mul_fold
      LRPX_CHECK_ARG(epi == LRPX_TC_EPI_MUL && a->ncol == 64 && a->ksize == 3, "folded filter columns: MUL epilogue, 64 columns, 3x3");
      p.fold = 1;
      p.taps = 3;
      p.bn = 3 * a->ncol;
    }
    if (epi == LRPX_TC_EPI_STORE_F32 && a->ncol > 256 && a->ncol % 256 && a->ncol % 64 == 0) p.bn = 64;
    LRPX_CHECK_ARG(p.fold || a->ncol % p.bn == 0, "ncol must be <= 256 or a multiple of 256 (STORE_F32: or of 64)");
    // plain GEMMs with few rows (the decoder's per-step GEMMs: 1216 x 1536 x 1536): 256-column tiles give fewer tiles
    // than SMs; 128-column tiles fill the machine (LRPX_TC_GEMM_BN=256 keeps the wide tiles)
    if (a->ksize == 1 && epi == LRPX_TC_EPI_STORE_F32 && p.bn == 256) {
      const char* env_bn = getenv("LRPX_TC_GEMM_BN");
      const long long m_tiles = ((long long)a->n_img * (a->h + 1) * (a->w + 1) + TC_BM - 1) / TC_BM;
      if (!(env_bn && atoi(env_bn) == 256) && m_tiles * (a->ncol / 256) < sm_count()) p.bn = 128;
    }
    p.out_c = a->ncol;
    p.n_valid = a->ncol;
    if (epi == LRPX_TC_EPI_STORE_F32 && a->out_pitch > 0) {
      LRPX_CHECK_ARG(a->n_valid > 0 && a->n_valid <= a->ncol && a->n_valid % 4 == 0 && a->out_pitch >= a->n_valid &&
                         a->out_pitch % 4 == 0, "STORE_F32: n_valid / out_pitch must be multiples of 4, n_valid <= ncol");
      p.out_c = a->out_pitch;
      p.n_valid = a->n_valid;
    }
  }
  p.num_n_tiles = p.fold ? 1 : a->ncol / p.bn;
  {
    int s = 0;
    while ((1LL << s) < p.num_n_tiles) ++s;
    p.nnt_sh = 31 + s;
    p.nnt_mul = (uint32_t)((((unsigned long long)1 << p.nnt_sh) + (unsigned long long)p.num_n_tiles - 1) / (unsigned long long)p.num_n_tiles);
  }
  cudaStream_t st = as_stream(stream);
  {
    const char* e2 = getenv("LRPX_TC_DEBUG");
    p.debug_flags = e2 ? atoi(e2) : 0;
    const char* e3 = getenv("LRPX_TC_SLEEP");
    p.sleep_ns = e3 ? atoi(e3) : 200;

  }
  {
    const char* env = getenv("LRPX_TC_SLAB");       // LRPX_TC_SLAB=0 falls back to one TMA tile per filter tap
    const bool want_slab = a->ksize == 3 && !(env && env[0] == '0');
    // EPI_MUL: results leave through a 16 KB staging area (1 KB per epilogue warp) and TMA tile stores
    const char* env_ts = getenv("LRPX_TC_TMASTORE");
    const bool tma_store = epi == LRPX_TC_EPI_MUL && !p.fold && !(env_ts && env_ts[0] == '0');
    const int reserve = tma_store ? TC_EPI_WARPS * 1024 : 0;
    // the pair decision up to the tile count (known after planning): it decides how much of B a CTA holds
    const char* env_cl = getenv("LRPX_TC_CLUSTER");             // LRPX_TC_CLUSTER=0: one CTA per cluster
    const bool want_cluster = !(env_cl && env_cl[0] == '0');
    const char* env_pair = getenv("LRPX_TC_PAIR");
    const bool pair_on = env_pair ? env_pair[0] != '0' : LRPX_TC_PAIR_DEFAULT;
    // error-compensated operands (K wrap: three times the K, hence three times the B tiles per accumulator tile): the
    // pair pays from 64 columns on — 224^2 64->64: 1.71 -> 1.52 ms, 112^2 128->64 un-pool: 0.84 -> 0.73 ms per 128 requests
    const int pair_min_bn = (env_pair && env_pair[0] == '2') ? 32 : (p.a_wrap ? 64 : 128);
    const char* env_pres = getenv("LRPX_TC_PAIR_RES");          // "0": plan the B residency as if each CTA held all of B
    bool pair_pre = want_cluster && pair_on && !p.fold && p.bn % 32 == 0 && p.bn >= pair_min_bn &&
                    (epi == LRPX_TC_EPI_MUL || epi == LRPX_TC_EPI_MUL_UNPOOL || epi == LRPX_TC_EPI_MULX ||
                     epi == LRPX_TC_EPI_MULX_UNPOOL) && sm_count() >= 2;
    const bool pair_res = pair_pre && !(env_pres && env_pres[0] == '0');
    if (want_slab && plan_slab(p, reserve, pair_res)) {
      p.half_rows = p.fold ? TC_BM - 2 : TC_BM;
      p.tile_out_rows = p.mh * p.half_rows;
      p.num_m_tiles = (p.m_total + p.tile_out_rows - 1) / p.tile_out_rows;
      if (pair_res && p.num_m_tiles < 2) {          // no pair after all: plan again with the whole B per CTA
        pair_pre = false;
        if (!plan_slab(p, reserve, false)) { set_error("slab planning failed"); return LRPX_E_INVALID; }
        p.tile_out_rows = p.mh * p.half_rows;
        p.num_m_tiles = (p.m_total + p.tile_out_rows - 1) / p.tile_out_rows;
      }
      p.tile_stride = p.tile_out_rows;
      p.walk = 0;
      p.tiles_per_cta = 0;
      const bool want_pair = pair_pre && p.num_m_tiles >= 2;
      p.a_group = 1;
      {
        // First layer: the three slabs of a tile in ONE ring stage (LRPX_TC_AGROUP=0: one stage per slab).  Its tiles are
        // 24 short MMAs; what bounds it is the issuers' and the producer's barrier traffic per tile (measured with the
        // timing switches: 0.19 ms per 128 requests with the epilogue reduced to the hand-back, 0.15 ms with neither MMAs
        // nor A traffic) — three wait / commit round trips per tile become one.
        const char* env_ag = getenv("LRPX_TC_AGROUP");
        const char* env_wk = getenv("LRPX_TC_WALK");            // the row walk (below) needs one stage per slab
        const bool walk_asked = env_wk && env_wk[0] == '1';
        const long long b_region = (long long)p.taps * p.kc_per_tap * p.bn * TC_BK * 2;
        const int budget = TC_SMEM_BYTES - 1024 - reserve;
        if (epi == LRPX_TC_EPI_INPUT3 && !(env_ag && env_ag[0] == '0') && !walk_asked && p.slab_mode == 3 && p.b_resident && !want_pair &&
            2LL * 3 * p.a_stage_bytes + b_region <= budget) {
          p.a_group = 3;
          p.a_stages = (int)((budget - b_region) / (3LL * p.a_stage_bytes));
          if (p.a_stages > TC_A_MAX_STAGES) p.a_stages = TC_A_MAX_STAGES;
          p.a_stage_bytes *= 3;
        }
      }
      {
        // four accumulator buffers where a tile's accumulators fit 128 TMEM columns (LRPX_TC_NBUF=2: never, =4: every
        // eligible layer; default: the first layer only, whose tiles are a round trip of barrier latencies long)
        const char* env_nb = getenv("LRPX_TC_NBUF");
        const bool fits = p.mh * p.bn <= 128 && !want_pair;
        const int want = env_nb ? atoi(env_nb) : (epi == LRPX_TC_EPI_INPUT3 ? 4 : 2);
        p.nbuf_log2 = (fits && want == 4) ? 2 : 1;
      }
      {
        // row walk for the wide first layer (LRPX_TC_WALK=1; OFF by default): tiles one image row apart, two of three slabs
        // reused.  Built on the hypothesis that the layer was bound by its 3x L2 -> SM re-fetch of A; measured on B200 it
        // is not (0.218 ms per 128 requests with the strided walk, 0.237 ms with the row walk: the tile time is a round trip
        // of barrier latencies, and the walk's tiles carry 225 instead of 252 rows) — kept as a tested switch
        const char* env_walk = getenv("LRPX_TC_WALK");
        if (epi == LRPX_TC_EPI_INPUT3 && env_walk && env_walk[0] == '1' && p.a_group == 1 && p.slab_mode == 3 && p.b_resident &&
            p.kc_per_tap == 1 && p.a_stages >= 4 && !want_pair && p.wp1 <= p.tile_out_rows && p.wp1 * 5 >= p.tile_out_rows * 4) {
          p.walk = 1;
          p.tile_stride = p.wp1;
          p.num_m_tiles = (p.m_total + p.tile_stride - 1) / p.tile_stride;
        }
      }
      CUtensorMap ma0, ma1, mb, mo;
      mo = CUtensorMap{};
      p.store_off = 0;
      if (tma_store) {
        const long long b_region = p.b_resident ? (long long)p.taps * p.kc_per_tap * p.bn * TC_BK * 2 / (want_pair ? 2 : 1)
                                                : (long long)p.b_stages * p.bn * TC_BK * 2;
        p.store_off = (int)((p.a_stages * (long long)p.a_stage_bytes + b_region + 1023) & ~1023LL);
        int rco = make_map_out(&mo, a->out, (uint64_t)p.m_total, (uint64_t)p.out_c);
        if (rco) return rco;
      }
      int rc = make_map_2d(&ma0, a->a, (uint64_t)p.m_total, (uint64_t)a_phys, (uint32_t)p.box0_rows);
      if (rc) return rc;
      rc = make_map_2d(&ma1, a->a, (uint64_t)p.m_total, (uint64_t)a_phys, (uint32_t)(p.box1_rows ? p.box1_rows : 8));
      if (rc) return rc;
      rc = make_map_2d(&mb, a->wt, (uint64_t)(epi == LRPX_TC_EPI_MUL && p.fold ? 3 * a->ncol : a->ncol),
                       (uint64_t)p.taps * a->cin, (uint32_t)p.bn);
      if (rc) return rc;
      // CTA pairs sharing the streamed B tiles through TMA multicast (halves the L2 -> SM weight traffic, which is
      // what bounds the 256/512-channel layers: ~12 TB/s of B re-fetches at 128-row tiles)
      CUtensorMap mbh = mb;
      p.cluster = 1;
      p.tiles_sched = p.num_m_tiles * p.num_n_tiles;
      // CTA pairs on ONE tcgen05.mma.cta_group::2 (M = 256 across the pair, each CTA holding bn/2 rows of B in its own
      // shared memory): halves the B operand reads per SM.  Measured per layer, A/B inside one process
      // (scripts/pair_ab.py, outputs bit-identical): 128-column layers -10 % (56^2 un-pool) and -20 % (112^2), 256-column
      // layers -4...9 %; the 64-column layers do NOT gain (224^2: +19 %, 112^2 un-pool: +-0: their tiles are short, K = 576 /
      // 1152, and the hand-over between the two CTAs costs more than the saved operand reads), so pairs start at 128 columns.
      // LRPX_TC_PAIR=0: off, =2: every width.
      p.pair = 0;
      if (want_pair) {
        p.pair = 1;
        p.cluster = 2;
        p.tiles_sched = p.num_n_tiles * 2 * ((p.num_m_tiles + 1) / 2);
        rc = make_map_2d(&mbh, a->wt, (uint64_t)a->ncol, (uint64_t)p.taps * a->cin, (uint32_t)(p.bn / 2));
        if (rc) return rc;
      } else if (want_cluster && !p.b_resident && p.bn >= 16 && sm_count() >= 2) {
        p.cluster = 2;
        p.tiles_sched = p.num_n_tiles * 2 * ((p.num_m_tiles + 1) / 2);
        rc = make_map_2d(&mbh, a->wt, (uint64_t)a->ncol, (uint64_t)p.taps * a->cin, (uint32_t)(p.bn / 2));
        if (rc) return rc;
      }
      int tiles = p.tiles_sched;
      int grid = tiles < sm_count() ? tiles : sm_count();
      if (p.cluster == 2) grid &= ~1;
      if (p.walk) {                     // contiguous runs: every CTA of the grid has at least one tile
        p.tiles_per_cta = (tiles + grid - 1) / grid;
        grid = (tiles + p.tiles_per_cta - 1) / p.tiles_per_cta;
      }
      switch (epi) {
        case LRPX_TC_EPI_FWD_GAIN: return launch_tc_slab<LRPX_TC_EPI_FWD_GAIN>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_MUL:
          if (p.fold) return launch_tc_slab<TC_EPI_MUL_FOLD>(ma0, ma1, mb, mbh, mo, p, grid, st);
          return launch_tc_slab<LRPX_TC_EPI_MUL>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_MUL_UNPOOL: return launch_tc_slab<LRPX_TC_EPI_MUL_UNPOOL>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_INPUT: return launch_tc_slab<LRPX_TC_EPI_INPUT>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_INPUT3:
          if (p.cam_rows) return launch_tc_slab<TC_EPI_INPUT3_CAM>(ma0, ma1, mb, mbh, mo, p, grid, st);
          return launch_tc_slab<LRPX_TC_EPI_INPUT3>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_MULX:
          if (p.mulx_simple) return launch_tc_slab<TC_EPI_MULX_S>(ma0, ma1, mb, mbh, mo, p, grid, st);
          return launch_tc_slab<LRPX_TC_EPI_MULX>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_MULX_UNPOOL:
          if (p.mulx_simple) return launch_tc_slab<TC_EPI_MULX_UNPOOL_S>(ma0, ma1, mb, mbh, mo, p, grid, st);
          return launch_tc_slab<LRPX_TC_EPI_MULX_UNPOOL>(ma0, ma1, mb, mbh, mo, p, grid, st);
        case LRPX_TC_EPI_FWDX:
          if (p.fwd_simple) return launch_tc_slab<TC_EPI_FWDX_SIMPLE>(ma0, ma1, mb, mbh, mo, p, grid, st);
          if (p.split && (p.idn || p.hd)) return launch_tc_slab<TC_EPI_FWDX_SPLIT_ADD>(ma0, ma1, mb, mbh, mo, p, grid, st);
          return launch_tc_slab<LRPX_TC_EPI_FWDX>(ma0, ma1, mb, mbh, mo, p, grid, st);
        default: return launch_tc_slab<LRPX_TC_EPI_STORE_F32>(ma0, ma1, mb, mbh, mo, p, grid, st);
      }
    }
  }
  LRPX_CHECK_ARG(epi != LRPX_TC_EPI_INPUT3 && !p.fold, "folded filter columns need the slab kernel (3x3, LRPX_TC_SLAB != 0)");
  p.slab_mode = 0; p.mh = 1; p.n_issuers = 1; p.cluster = 1; p.half_rows = TC_BM; p.tile_out_rows = TC_BM;
  p.num_m_tiles = (p.m_total + TC_BM - 1) / TC_BM;
  const int stage_bytes = TC_A_BYTES + p.bn * TC_BK * 2;
  p.stages = (TC_SMEM_BYTES - 1024) / stage_bytes;
  if (p.stages > TC_MAX_STAGES) p.stages = TC_MAX_STAGES;
  LRPX_CHECK_ARG(p.stages >= 2, "tile does not fit in shared memory");

  CUtensorMap ma, mb;
  int rc = make_map_2d(&ma, a->a, (uint64_t)p.m_total, (uint64_t)a_phys, TC_BM);
  if (rc) return rc;
  rc = make_map_2d(&mb, a->wt, (uint64_t)a->ncol, (uint64_t)p.taps * a->cin, (uint32_t)p.bn);
  if (rc) return rc;

  int tiles = p.num_m_tiles * p.num_n_tiles;
  int grid = tiles < sm_count() ? tiles : sm_count();
  switch (epi) {
    case LRPX_TC_EPI_FWD_GAIN: return launch_tc<LRPX_TC_EPI_FWD_GAIN>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_MUL: return launch_tc<LRPX_TC_EPI_MUL>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_MUL_UNPOOL: return launch_tc<LRPX_TC_EPI_MUL_UNPOOL>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_INPUT: return launch_tc<LRPX_TC_EPI_INPUT>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_FEAT: return launch_tc<LRPX_TC_EPI_FEAT>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_FEAT_DIV: return launch_tc<LRPX_TC_EPI_FEAT_DIV>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_MULX:
      if (p.mulx_simple) return launch_tc<TC_EPI_MULX_S>(ma, mb, p, grid, st);
      return launch_tc<LRPX_TC_EPI_MULX>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_MULX_UNPOOL:
      if (p.mulx_simple) return launch_tc<TC_EPI_MULX_UNPOOL_S>(ma, mb, p, grid, st);
      return launch_tc<LRPX_TC_EPI_MULX_UNPOOL>(ma, mb, p, grid, st);
    case LRPX_TC_EPI_FWDX:
      if (p.fwd_simple) return launch_tc<TC_EPI_FWDX_SIMPLE>(ma, mb, p, grid, st);
      if (p.split && (p.idn || p.hd)) return launch_tc<TC_EPI_FWDX_SPLIT_ADD>(ma, mb, p, grid, st);
      return launch_tc<LRPX_TC_EPI_FWDX>(ma, mb, p, grid, st);
    default: return launch_tc<LRPX_TC_EPI_STORE_F32>(ma, mb, p, grid, st);
  }
}

extern "C" int lrpx_tc_gemm_bf16_f32(const void* a, const void* wt, float* out, int m, int n, int k, void* stream) {
  LRPX_CHECK_ARG(a && wt && out && m > 0 && n > 0 && k > 0, "bad argument");
  LRPX_CHECK_ARG(k % TC_BK == 0 && n % 32 == 0 && (n <= 256 || n % 256 == 0), "unsupported GEMM shape");
  // one PF "block" of m rows (h = 0, w = m - 1): the STORE_F32 epilogue writes every in-range row
  lrpx_tc_conv_args g{};
  g.n_img = 1; g.h = 0; g.w = m - 1; g.cin = k; g.ncol = n; g.ksize = 1; g.epilogue = LRPX_TC_EPI_STORE_F32;
  g.a = a; g.wt = wt; g.out = out;
  return lrpx_tc_conv(&g, stream);
}
