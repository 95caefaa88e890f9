/*
 * lrpx.h — C ABI of liblrpx.so: layer-wise relevance propagation (LRP) kernels for sm_100a (B200).
 *
 * This is the drop-in boundary for the LRP hot path of SunJiamei/LRP-imagecaptioning-pytorch.
 * The reference has no FFI of its own (pure Python, SURVEY.md §8b); each entry point below
 * replaces the arithmetic of one reference call site, cited as `file:line` relative to the
 * reference repository.  The Python host layer (lrp-imagecaptioning-pytorch_b200/LRPtools, models)
 * keeps the reference's own signatures and binds these symbols with ctypes (INTEGRATION.md).
 *
 * Conventions
 *   - every function returns 0 on success, <0 on error (LRPX_E_*); lrpx_last_error() gives a
 *     thread-local message.  No exceptions cross the boundary.
 *   - all pointers are DEVICE pointers owned by the caller; nothing is allocated or freed here,
 *     nothing synchronises; work is enqueued on `stream` (a cudaStream_t passed as void*).
 *   - "f32" entry points: NCHW / row-major fp32, the reference's own layout and precision
 *     (parity path, rtol 1e-4 / atol 1e-6 against the oracle).
 *   - "tc" entry points: NHWC bf16 operands, fp32 accumulation on tcgen05 tensor cores
 *     (throughput path; tolerance stated in tests/test_tc_parity.py).
 *   - the library has no mutable global state apart from a once-initialised driver entry point.
 */
#ifndef LRPX_H_
#define LRPX_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LRPX_OK 0
#define LRPX_E_INVALID (-1)   /* bad argument (null pointer, unsupported shape, ...) */
#define LRPX_E_CUDA (-2)      /* a CUDA runtime/driver call failed                    */
#define LRPX_E_UNSUPPORTED (-3)

/* constants of LRPtools/utils.py:7-14 */
#define LRPX_EPSILON 0.01f
#define LRPX_Z_EPSILON 1e-7f
#define LRPX_RELEVANCE_RECT (-1e-6f)

const char* lrpx_last_error(void);
int lrpx_version(void);
/* compute capability major*10+minor of the current device, or <0 */
int lrpx_device_cc(void);

/* ---------------------------------------------------------------------------------------------
 * Conv2d relevance, fp32 NCHW (LRPtools/lrp_modules.py:56-170 + LRPtools/utils.py:16-31)
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int n, cin, h, w;        /* input  (n, cin, h, w)                 */
  int cout, kh, kw;        /* weight (cout, cin, kh, kw), groups==1 */
  int stride_h, stride_w, pad_h, pad_w, dil_h, dil_w;
} lrpx_conv_shape;

enum { LRPX_NET_POS = 0, LRPX_NET_NEG = 1, LRPX_NET_PLAIN = 2 };

/* K1: z = net(a)  then  s = r_out / (z + 1e-7*[z==0])            (utils.py:16-18,26-27)
 *   net POS : z = conv(a+,W+) + conv(a-,W-)                      (PosNetConv, lrp_modules.py:81-84)
 *   net NEG : z = conv(a-,W+) + conv(a+,W-)                      (NegNetConv, lrp_modules.py:111-114)
 *   net PLAIN (epsilon rule, "parity unpinned" for conv): zeros of `a` count as -1e-6, z = conv(a,W),
 *             s = r_out / (z + 0.01*sign z, 0 -> 0.01)            (Linear rule, lrp_modules.py:13-22)
 * bias may be NULL (ignore_bias=True); otherwise z += bias (clamp(b,min=0)+clamp(b,max=0) == b).
 * z_out may be NULL; when given it receives z (used for conservation reports). */
int lrpx_conv_rule_s_f32(const float* a, const float* w, const float* bias, const float* r_out, float* s,
                         float* z_out, const lrpx_conv_shape* shp, int net, void* stream);

/* K2: r_in (+)= scale * a (.) dgrad(net, s)                      (utils.py:29-30: Z.backward(S); X*X.grad)
 * accumulate != 0 adds into r_in (used for  alpha*R_pos - beta*R_neg, lrp_modules.py:134-146). */
int lrpx_conv_rule_rin_f32(const float* a, const float* w, const float* s, float* r_in,
                           const lrpx_conv_shape* shp, int net, float scale, int accumulate, void* stream);

/* plain forward conv (+bias, optional ReLU) used to produce the saved layer inputs (lrp_wrapper.py:70) */
int lrpx_conv_forward_f32(const float* a, const float* w, const float* bias, float* out,
                          const lrpx_conv_shape* shp, int relu, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Linear epsilon rule in GEMM form, fp32 row-major (LRPtools/lrp_modules.py:9-37)
 *   a (n,in)  w (out,in)  r_out (n,out)  ->  r_in (n,in);  a is NOT modified (the reference fills
 *   its zeros with -1e-6 in place, Q9; here the fill is applied on the fly).
 * ------------------------------------------------------------------------------------------- */
int lrpx_linear_eps_f32(const float* a, const float* w, const float* bias, const float* r_out, float* r_in,
                        float* s_workspace /* n*out floats */, int n, int in_features, int out_features,
                        int ignore_bias, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Pooling (LRPtools/lrp_modules.py:172-195), fp32 NCHW
 * ------------------------------------------------------------------------------------------- */
typedef struct { int n, c, h, w, kh, kw, stride_h, stride_w, pad_h, pad_w; } lrpx_pool_shape;

/* forward max-pool with PyTorch's argmax (flat index inside the (h,w) plane, first max in scan
 * order, NaN wins) — the bit-exact index contract of SURVEY.md §8(a4). y and/or idx may be NULL. */
int lrpx_maxpool_forward_f32(const float* x, float* y, int64_t* idx, const lrpx_pool_shape* shp, void* stream);
/* winner-take-all: r_in = x * scatter(r_out / (max + 1e-7*[max==0])) — gather form, deterministic */
int lrpx_maxpool_wta_f32(const float* x, const float* r_out, float* r_in, const lrpx_pool_shape* shp, void* stream);
/* avg-pool: r_in = x * sum_windows( s / (kh*kw) ),  s = r_out / (avg + 1e-7*[avg==0])
 * (count_include_pad=True, ceil_mode=False — the nn.AvgPool2d defaults) */
int lrpx_avgpool_prop_f32(const float* x, const float* r_out, float* r_in, const lrpx_pool_shape* shp, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Element-wise rules, fp32
 * ------------------------------------------------------------------------------------------- */
/* BatchNorm abs-ratio, lrp_modules.py:204-215 (x is (n,c,hw)) */
int lrpx_bn_absratio_f32(const float* x, const float* r_out, float* r_in, const float* running_mean,
                         const float* running_var, const float* gamma, const float* beta, float eps, int n,
                         int c, int hw, void* stream);
/* residual Add proportional split, lrp_modules.py:262-275 */
int lrpx_add_split_f32(const float* x1, const float* x2, const float* r_out, float* r1, float* r2, size_t count,
                       void* stream);
/* ReLU non-identity rule, lrp_modules.py:48-54: r_in = r_out * [x > 0] */
int lrpx_relu_mask_f32(const float* x, const float* r_out, float* r_in, size_t count, void* stream);
/* utils.normalize_relevance (utils.py:55-64), row-wise over the last dim, temperature as given */
int lrpx_normalize_relevance_f32(const float* x, float* y, int rows, int cols, float temperature, void* stream);
/* sum of a buffer in double precision (conservation reports: sum R_in vs sum R_out); out is 1 double */
int lrpx_sum_f64(const float* x, size_t count, double* out, void* stream);

/* The explainers' NAMED vector rules (the batched decoder kernels below fuse the same arithmetic; these serve the
 * reference's own method names as CUDA entry points):
 * lrp_linear_eps (gridTDmodel.py:744-765 / :522-547, aoamodel.py:532-557,785-810):
 *   r_in[j] = x[j] * sum_k W[k][j] * r_out[k] / stab(z[k]),  stab(z) = z + 0.01*sign(z), 0 -> 0.01;
 *   z == NULL means forward_output=False in the reference: z = W x is recomputed (without bias).
 *   W is (n_out, n_in) row-major.  workspace: lrpx_lrp_linear_eps_workspace_bytes(n_out, n_in) bytes. */
size_t lrpx_lrp_linear_eps_workspace_bytes(int n_out, int n_in);
int lrpx_lrp_linear_eps_f32(const float* r_out, const float* x, const float* z, const float* W, float* r_in, int n_out,
                            int n_in, void* workspace, size_t workspace_bytes, void* stream);
/* lrp_mha (aoamodel.py:812-862): value relevance of ONE head,
 *   r_value[p][c] = value[p][c] * alpha[head][p] * r_context[c] / stab(context[c]) for c in head's d_k slice, else 0
 *   alpha (num_head, P), value / r_value (P, H), r_context / context (H). */
int lrpx_lrp_mha_f32(const float* alpha, const float* value, const float* r_context, const float* context, float* r_value,
                     int P, int H, int num_head, int head_idx, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Decoder relevance, fp32 (models/gridTDmodel.py:1014-1135, models/aoamodel.py:812-862,1064-1156),
 * batched over Q explanation requests (image b_q, target word t_q).
 * Saved-state tensors are those of get_hidden_parameters (gridTDmodel.py:933-1012), stacked over
 * B images and padded to T steps:   name[b][t][...]  row-major.
 * ------------------------------------------------------------------------------------------- */
/* flags of the decoder entry points */
#define LRPX_DEC_TC_GEMM 1   /* run the GEMMs on tcgen05 tensor cores as error-compensated bf16x3 (a_hi*w_hi + a_hi*w_lo +
                                a_lo*w_hi, fp32 accumulate: ~2^-16 relative per product) instead of fp32 CUDA cores */
#define LRPX_DEC_W3_READY 4  /* with LRPX_DEC_TC_GEMM, the three LRP decoders: the prepared (split bf16) copies of the weight
                                matrices that an EARLIER call wrote into this same `workspace` are still valid — same
                                argument dimensions (the workspace layout depends on them), same weight values — and are
                                not rebuilt (four conversion kernels per call).  The caller owns that guarantee. */

typedef struct {
  int B, T, H, E, P, C, V, Q;
  int flags, reserved_;    /* LRPX_DEC_* */
  /* per image */
  const float* feat;      /* (B,P,C)  encoder output, pixel-major (NHWC)      gridTDmodel.py:1029-1030 */
  const float* avg;       /* (B,C)                                                         :941       */
  const float* A_pre;     /* (B,P,H)  1x1 projector output before ReLU                      :944,:950  */
  const float* A;         /* (B,P,H)  after ReLU                                            :945-949   */
  const float* glob_pre;  /* (B,E)                                                          :946       */
  /* per image and step */
  const float* x1;        /* (B,T,H+2E)  [h2_prev | glob | emb]                              :980,:995  */
  const float* x2;        /* (B,T,2H)    [ctx_hat | h1]                                      :987,:996  */
  const float* h1;        /* (B,T+1,H) row 0 = zeros                                         :1000      */
  const float* c1;        /* (B,T+1,H) */
  const float* h2;        /* (B,T+1,H) */
  const float* c2;        /* (B,T+1,H) */
  const float* g1;        /* (B,T,H) pre-tanh cell candidate                                 :1002      */
  const float* i1;        /* (B,T,H) sigmoid(input gate) */
  const float* f1;        /* (B,T,H) */
  const float* g2;
  const float* i2;
  const float* f2;
  const float* st;        /* (B,T,H) sentinel                                                :1010      */
  const float* ctx;       /* (B,T,H) */
  const float* ctx_hat;   /* (B,T,H) */
  const float* alpha;     /* (B,T,P) */
  const float* beta;      /* (B,T)   */
  const float* pred;      /* (B,T,V) logits                                                  :997       */
  /* weights */
  const float* W_g1;      /* (H, 2H+2E) = [W_ih | W_hh] rows of gate g of AdaLSTM            :1019-1021 */
  const float* W_g2;      /* (H, 3H)    same for LanguageLSTM                                :1022-1024 */
  const float* W_fc;      /* (V, H)                                                          :735       */
  const float* W_glob;    /* (E, C) global_img_feature_proj.weight                           :1119      */
  const float* W_proj;    /* (H, C) img_projector.weight squeezed                            :1128      */
  /* requests */
  const int32_t* req_img;   /* (Q) image index b_q                 */
  const int32_t* req_t;     /* (Q) target step t_q  (0 <= t_q < T) */
  const int32_t* req_word;  /* (Q) vocabulary id of the explained word = tokens[b_q][t_q+1]  :1017 */
  /* outputs */
  float* r_feat;            /* (Q,P,C) relevance of the encoder output, pixel-major          :1133 */
  float* r_words;           /* (Q,T)   normalised linguistic relevance, entries > t_q are 0  :1129-1132 */
  float* r_words_raw;       /* (Q,T)   before the max-abs normalisation (may be NULL)        */
} lrpx_gridtd_args;

size_t lrpx_gridtd_decoder_workspace_bytes(const lrpx_gridtd_args* args);
int lrpx_gridtd_decoder_lrp_f32(const lrpx_gridtd_args* args, void* workspace, size_t workspace_bytes, void* stream);

typedef struct {
  int B, T, H, E, P, C, V, Q, num_head;
  int flags;               /* LRPX_DEC_* */
  const float* feat;      /* (B,P,C)                                   aoamodel.py:1079-1080 */
  const float* A_pre;     /* (B,P,H)                                              :1006      */
  const float* A;         /* (B,P,H)                                              :1005      */
  const float* glob;      /* (B,H) mean over pixels of A                          :1007      */
  const float* value;     /* (B,P,H) decoder_v_proj(A)                            :1009      */
  const float* x;         /* (B,T,E+H) [emb | glob]                               :1030,:1042 */
  const float* h;         /* (B,T+1,H) */
  const float* c;         /* (B,T+1,H) */
  const float* g;         /* (B,T,H) */
  const float* i;         /* (B,T,H) */
  const float* ctx;       /* (B,T,H) attention output                             :1057      */
  const float* caoa;      /* (B,T,H) sigmoid(gate)*linear                         :1059      */
  const float* caoa_lin;  /* (B,T,H) decoder_aoa_linear(ctx)                      :1061      */
  const float* alpha;     /* (B,T,heads,P)                                        :1046      */
  const float* pred;      /* (B,T,V) */
  const float* W_g;       /* (H, E+2H) gate-g rows [W_ih | W_hh]                  :1072-1074 */
  const float* W_fc;      /* (V,H) */
  const float* W_aoa;     /* (H,H) decoder_aoa_linear.weight                      :1110      */
  const float* W_v;       /* (H,H) decoder_v_proj.weight                          :1144      */
  const float* W_proj;    /* (H,C) */
  const int32_t* req_img;
  const int32_t* req_t;
  const int32_t* req_word;
  const int32_t* req_head;  /* (Q) head_idx                                       :1112-1113 */
  float* r_feat;            /* (Q,P,C) */
  float* r_words;           /* (Q,T) */
  float* r_words_raw;
} lrpx_aoa_args;

size_t lrpx_aoa_decoder_workspace_bytes(const lrpx_aoa_args* args);
int lrpx_aoa_decoder_lrp_f32(const lrpx_aoa_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* ExplainAdaptiveAttention.explain_caption_wordt (models/adaptiveattention.py:679-771): the single-LSTM adaptive
 * attention decoder.  Saved state = get_hidden_parameters (:626-677), stacked over B images, padded to T steps. */
typedef struct {
  int B, T, H, E, P, C, V, Q;
  int flags, reserved_;    /* LRPX_DEC_* */
  /* per image */
  const float* feat;      /* (B,P,C)  encoder output, pixel-major                            adaptiveattention.py:748-749 */
  const float* avg;       /* (B,C)    mean feature = forward_input of the global rule                       :744       */
  const float* z_proj;    /* (B,P,H)  feat @ W_proj^T WITHOUT bias (forward_output=False)                   :762       */
  const float* A;         /* (B,P,H)  relu(z_proj + bias)                                                   :633       */
  const float* z_glob;    /* (B,E)    avg @ W_glob^T WITHOUT bias (forward_output=False)                    :745       */
  /* per image and step */
  const float* x;         /* (B,T,2E) [emb | glob]                                                          :649,:663  */
  const float* h;         /* (B,T+1,H) row 0 = zeros                                                        :667       */
  const float* c;         /* (B,T+1,H) */
  const float* g;         /* (B,T,H) pre-tanh cell candidate                                                :669       */
  const float* i;         /* (B,T,H) sigmoid(input gate) */
  const float* f;         /* (B,T,H) */
  const float* st;        /* (B,T,H) sentinel                                                               :672       */
  const float* ctx;       /* (B,T,H) */
  const float* ctx_hat;   /* (B,T,H) */
  const float* alpha;     /* (B,T,P) */
  const float* beta;      /* (B,T)   */
  const float* pred;      /* (B,T,V) logits                                                                 :664       */
  /* weights */
  const float* W_g;       /* (H, 2E+H) = [W_ih | W_hh] rows of gate g of AdaLSTM                            :685-687   */
  const float* W_fc;      /* (V, H)                                                                         :523       */
  const float* W_glob;    /* (E, C)                                                                         :746       */
  const float* W_proj;    /* (H, C)                                                                         :763       */
  /* requests */
  const int32_t* req_img;   /* (Q) */
  const int32_t* req_t;     /* (Q) 0 <= t_q < T */
  const int32_t* req_word;  /* (Q) tokens[b_q][t_q+1]                                                       :682       */
  /* outputs */
  float* r_feat;            /* (Q,P,C)                                                                      :768       */
  float* r_words;           /* (Q,T)  normalised, entries > t_q are 0                                       :764-767   */
  float* r_words_raw;       /* (Q,T)  may be NULL */
} lrpx_adaptive_args;

size_t lrpx_adaptive_decoder_workspace_bytes(const lrpx_adaptive_args* args);
int lrpx_adaptive_decoder_lrp_f32(const lrpx_adaptive_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Gradient-family explainers, decoder part (SURVEY.md §8 f4): the reference's hand-written backward pass of the
 * decoder with the attention weights and gates held constant, batched over Q requests like the relevance above.
 *   gridTD: ExplainGridTDGradient.explain_caption_wordt (gridTDmodel.py:1424-1508); LRPX_DEC_GUIDED adds the guided
 *           variant's mask d_feat[feat <= 0] = 0 (ExplainiGridTDGuidedGradient, :1663-1674)
 *   AoA:    ExplainAOAGradient.explain_caption_wordt (aoamodel.py:1435-1499) with gradient_mha (:1415-1433)
 * Saved state: that of get_hidden_parameters (:1323-1422 / aoamodel.py:1309-1375) — the relevance state plus the output
 * gates and the sentinel gate (lrpx_lstm_step_args.o / .sg) — stacked over B images, padded to T steps.
 * ------------------------------------------------------------------------------------------- */
#define LRPX_DEC_GUIDED 2

typedef struct {
  int B, T, H, E, P, C, V, Q;
  int flags, reserved_;    /* LRPX_DEC_TC_GEMM | LRPX_DEC_GUIDED */
  const float* feat;      /* (B,P,C) encoder output, pixel-major: the guided mask (NULL otherwise)   :1674 */
  const float* c1;        /* (B,T+1,H) AdaLSTM cell states, row 0 = zeros                            :1401 */
  const float* c2;        /* (B,T+1,H) LanguageLSTM                                                  :1411 */
  const float* g1;        /* (B,T,H) pre-tanh cell candidate (the kernels take tanh)                 :1404,:1408 */
  const float* i1;        /* (B,T,H) sigmoid(input gate)                                             :1406 */
  const float* f1;
  const float* o1;        /* (B,T,H) sigmoid(output gate)                                            :1409 */
  const float* g2;
  const float* i2;
  const float* f2;
  const float* o2;
  const float* sg;        /* (B,T,H) sigmoid(x_gate(x) + h_gate(h)), the sentinel gate               :1381,:1394 */
  const float* alpha;     /* (B,T,P) */
  const float* beta;      /* (B,T)   */
  const float* W1;        /* (4H, H+2E) AdaLSTM weight_ih: columns [h2 | glob | emb]                  :1495 */
  const float* W2;        /* (4H, 3H)   LanguageLSTM [weight_ih | weight_hh]: columns [ctx_hat | h1 | h2]  :1474-1475 */
  const float* W_fc;      /* (V,H)                                                                   :1459 */
  const float* W_glob;    /* (E,C)                                                                   :1499 */
  const float* W_proj;    /* (H,C)                                                                   :1502 */
  const int32_t* req_img;   /* (Q) */
  const int32_t* req_t;     /* (Q) 0 <= t_q < T */
  const int32_t* req_word;  /* (Q) tokens[b_q][t_q+1]                                                :1427 */
  float* d_feat;            /* (Q,P,C) gradient with respect to the encoder output, pixel-major      :1507 */
  float* r_words;           /* (Q,T) sum over the embedding of d logits / d emb_i, max-abs normalised :1503-1506 */
  float* r_words_raw;       /* (Q,T) before the normalisation (may be NULL) */
} lrpx_gridtd_grad_args;

size_t lrpx_gridtd_decoder_grad_workspace_bytes(const lrpx_gridtd_grad_args* args);
int lrpx_gridtd_decoder_grad_f32(const lrpx_gridtd_grad_args* args, void* workspace, size_t workspace_bytes, void* stream);

typedef struct {
  int B, T, H, E, P, C, V, Q, num_head;
  int flags;               /* LRPX_DEC_TC_GEMM */
  const float* c;         /* (B,T+1,H)                                             aoamodel.py:1363 */
  const float* g;         /* (B,T,H) pre-tanh cell candidate                                  :1366 */
  const float* i;         /* (B,T,H) gate activations                                         :1368-1371 */
  const float* f;
  const float* o;
  const float* caoa_gate; /* (B,T,H) decoder_aoa_linear_gate(h), before the sigmoid           :1375 */
  const float* caoa_lin;  /* (B,T,H) decoder_aoa_linear(ctx)                                  :1374 */
  const float* alpha;     /* (B,T,heads,P)                                                    :1361 */
  const float* W_g;       /* (4H, E+2H) LanguageLSTM [weight_ih | weight_hh]: columns [emb | glob | h]   :1486-1487 */
  const float* W_fc;      /* (V,H) */
  const float* W_aoa;     /* (H,H) decoder_aoa_linear.weight                                  :1469 */
  const float* W_gate;    /* (H,H) decoder_aoa_linear_gate.weight                             :1470 */
  const float* W_v;       /* (H,H) decoder_v_proj.weight                                      :1490 */
  const float* W_proj;    /* (H,C)                                                            :1493 */
  const int32_t* req_img;
  const int32_t* req_t;
  const int32_t* req_word;
  const int32_t* req_head;  /* (Q) head_idx                                                   :1472 */
  float* d_feat;            /* (Q,P,C) */
  float* r_words;           /* (Q,T) */
  float* r_words_raw;
} lrpx_aoa_grad_args;

size_t lrpx_aoa_decoder_grad_workspace_bytes(const lrpx_aoa_grad_args* args);
int lrpx_aoa_decoder_grad_f32(const lrpx_aoa_grad_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* ExplainAdaptiveGradient.explain_caption_wordt (adaptiveattention.py:965-1021; the guided variant :1100-1163 differs
 * only by masks that never fire): the attention / sentinel split is applied at the explained step only, the loop walks
 * the single AdaLSTM. */
typedef struct {
  int B, T, H, E, P, C, V, Q;
  int flags, reserved_;    /* LRPX_DEC_TC_GEMM */
  const float* c;         /* (B,T+1,H)                                              adaptiveattention.py:952 */
  const float* g;         /* (B,T,H) pre-tanh cell candidate                                    :955,:959 */
  const float* i;         /* (B,T,H) gate activations                                           :957-960  */
  const float* f;
  const float* o;
  const float* sg;        /* (B,T,H) sigmoid(x_gate(x) + h_gate(h)), the sentinel gate          :941,:946 */
  const float* alpha;     /* (B,T,P) */
  const float* beta;      /* (B,T)   */
  const float* W_g;       /* (4H, 2E+H) AdaLSTM [weight_ih | weight_hh]: columns [emb | glob | h]  :1007-1008 */
  const float* W_fc;      /* (V,H) */
  const float* W_glob;    /* (E,C)                                                              :1011 */
  const float* W_proj;    /* (H,C)                                                              :1015 */
  const int32_t* req_img;
  const int32_t* req_t;
  const int32_t* req_word;
  float* d_feat;          /* (Q,P,C) */
  float* r_words;         /* (Q,T) */
  float* r_words_raw;
} lrpx_adaptive_grad_args;

size_t lrpx_adaptive_decoder_grad_workspace_bytes(const lrpx_adaptive_grad_args* args);
int lrpx_adaptive_decoder_grad_f32(const lrpx_adaptive_grad_args* args, void* workspace, size_t workspace_bytes, void* stream);

/* Grad-CAM (gridTDmodel.py:1760-1771, aoamodel.py:1676-1689), one map per request:
 *   weights[c] = mean_p grads[q][p][c];  cam[p] = relu(sum_c feat[img(q)][p][c] * weights[c]);  out[q][p] = cam[p] / (max cam + 1e-6)
 * feat (B,P,C) and grads (Q,P,C) pixel-major; req_img (Q) or NULL = identity; out (Q,P). */
int lrpx_grad_cam_f32(const float* feat, const float* grads, const int32_t* req_img, float* out, int Q, int P, int C,
                      void* stream);

/* Guided Grad-CAM (gridTDmodel.py:1812-1833): out[q][c][y][x] = g[q][c][y][x] * (Kh cam_q Kw^T)[y][x].  g / out (Q,C,H,W)
 * (may alias), cam (Q,h,w), Kh (H,h) and Kw (W,w): skimage.transform.pyramid_expand along one axis as a matrix (bilinear
 * resize then Gaussian smoothing, both separable), built by the host (models/_gradient.py::expand_operator). */
int lrpx_cam_expand_mul_f32(const float* g, const float* cam, const float* Kh, const float* Kw, float* out, int Q, int C,
                            int h, int w, int H, int W, void* stream);

/* Guided Grad-CAM's expansion along y (gridTDmodel.py:1826-1828), the first half of Kh cam_q Kw^T:
 *   out[q][y][j] = sum_i Kh[y][i] * cam[q][i][j]   (fmaf over i = 0..h-1, lrpx_cam_expand_mul_f32's order)
 * cam (Q,h,w), Kh (H,h), out (Q,H,w).  The tensor-core chain's INPUT3 epilogue applies the x half (cam_rows / cam_kw
 * of lrpx_tc_conv_args) where it forms the image gradient, so the guided gradient is never stored un-multiplied. */
int lrpx_cam_expand_rows_f32(const float* cam, const float* Kh, float* out, int Q, int h, int w, int H, void* stream);

/* lrp_tune weights, batched (gridTDmodel.py:549-578, aoamodel.py:597-626, utils.py:55-64):
 *   w = argmax logits[b]; if is_stop[w] -> weights 1; else r = fc-row eps rule, split to h / ctx,
 *   weights = r / max|r| + 1.   No host synchronisation; is_stop is a device byte mask (V). */
int lrpx_fc_lrp_weights_f32(const float* logits, const float* h, const float* ctx, const float* W_fc,
                            const uint8_t* is_stop, float* w_ctx, float* w_h, int32_t* argmax_out /* may be NULL */,
                            int B, int V, int H, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Beam search bookkeeping on the device (SURVEY §8 f1): one step of GridTDModel.beam_search
 * (models/gridTDmodel.py:400-478; same loop in aoamodel.py:405-485 and adaptiveattention.py:370-447) for B images
 * with k beam slots each.  Slots [0, n_alive[b]) of image b are its unfinished beams in the reference's order.
 * A step takes the logits of the B*k rows and
 *   - adds log_softmax(logits[r]) to the running score of every alive row (row 0 only at step 0, :436-439),
 *   - selects the n_alive best (row, word) pairs in descending order, ties to the lower flat index (:440),
 *   - moves pairs ending in end_id to the completed list (sequence incl. <end>, score; :449-452),
 *   - compacts the others into the new alive slots: seqs, scores, prev_words, and src_row[b*k+j] = the global row
 *     whose recurrent state slot j continues (:455-462) — dead slots point at themselves.
 * No host synchronisation; the caller reads seqs / comp_* once after the last step (:463-468).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int B, k, V, L;          /* k <= 8 slots per image, L = max_cap_length steps (L + 1 <= 64 tokens per sequence) */
  int step, end_id;        /* 0 <= step < L */
  const float* logits;     /* (B*k, V) */
  float* scores;           /* (B,k)     running log-probabilities, zero before step 0 */
  int32_t* n_alive;        /* (B)       k before step 0 */
  int32_t* seqs;           /* (B,k,L+1) alive sequences, column 0 = <start> */
  int32_t* comp_seqs;      /* (B,k,L+1) completed sequences in completion order */
  int32_t* comp_len;       /* (B,k)     their token counts */
  float* comp_scores;      /* (B,k) */
  int32_t* n_comp;         /* (B)       0 before step 0 */
  int64_t* prev_words;     /* (B*k)     input words of the next step (int64: an embedding index) */
  int32_t* src_row;        /* (B*k) */
} lrpx_beam_args;

int lrpx_beam_step(const lrpx_beam_args* args, void* stream);

/* dst[e][row][0:width[e]] = src[e][src_row[row]][0:width[e]] for every pair e (state[beam_idx], gridTDmodel.py:459);
 * dst and src of a pair must be different buffers. */
#define LRPX_BEAM_GATHER_MAX 8
typedef struct {
  int n_rows, n_pairs;
  const int32_t* src_row;
  float* dst[LRPX_BEAM_GATHER_MAX];
  const float* src[LRPX_BEAM_GATHER_MAX];
  long long ld_dst[LRPX_BEAM_GATHER_MAX];
  long long ld_src[LRPX_BEAM_GATHER_MAX];
  int width[LRPX_BEAM_GATHER_MAX];
} lrpx_beam_gather_args;

int lrpx_beam_gather_f32(const lrpx_beam_gather_args* args, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Patch ablation (SURVEY §8 f3): EvaluationExperiments.block_image (evaluation.py:57-80) batched over Q requests.
 * spatial relevance = channel mean of the request's heat-map (:128-129); the k patches (patch x patch pixels) with the
 * largest relevance sums are blanked: mask = 0 there, 1 elsewhere (:73-80); masked = mask * images[req_img[q]] (:130).
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int Q, C, H, W;          /* heat-maps (Q,C,H,W) */
  int patch, k;            /* evaluation.py:55-56: patch_size 8, num_delete_patches 20 */
  int img_c, reserved_;    /* channels of `images` */
  const float* heat;
  const float* images;     /* (B,img_c,H,W) or NULL */
  const int32_t* req_img;  /* (Q) image of each request, NULL = identity */
  float* mask;             /* (Q,H,W) or NULL */
  float* masked;           /* (Q,img_c,H,W) or NULL */
} lrpx_block_image_args;

int lrpx_block_image_f32(const lrpx_block_image_args* args, void* stream);

/* Bounding-box correctness of an explanation (EvaluationExperiments._calculate_overlaped_pixels + _project_maxabs,
 * evaluation.py:310-342, as bbox_experiment applies them, :398-431), batched over Q requests:
 *   m = maxabs-normalised mean over the channels of max(sign * heat, 0); for every threshold: m[m <= thr] = 0;
 *   ratio = min(1, sum(m inside the box) / sum(m)), 0 when sum(m) == 0.        Boxes are (x0, y0, x1, y1), ends exclusive. */
typedef struct {
  int Q, C, H, W;
  int n_thr, max_boxes;    /* max_boxes <= 8 */
  float sign;              /* +1, or -1 for the 'neg' explanation types (:398-401) */
  int inplace_quirk;       /* 1: like the reference, whose thresholding mutates the map (:324-326), every (box, threshold)
                              pair in bbox_experiment's loop order (:419-431) sees the largest threshold applied before
                              it; 0: every pair is evaluated on the fresh map */
  const float* heat;       /* (Q,C,H,W) */
  const float* thresholds; /* (n_thr)   evaluation.py:425 uses 0, 0.1, ..., 0.9 */
  const int32_t* boxes;    /* (Q,max_boxes,4) */
  const int32_t* n_boxes;  /* (Q) boxes in use per request, NULL = max_boxes */
  float* ratio;            /* (Q,max_boxes,n_thr); unused box slots are set to 0 */
} lrpx_bbox_args;

int lrpx_bbox_ratio_f32(const lrpx_bbox_args* args, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Explainer forward (the producer of the saved state above): fused element-wise steps of
 * ExplainGridTDAttention.get_hidden_parameters (gridTDmodel.py:933-1012).  Row strides ("ld_*", in
 * elements) let the kernels write straight into the (B, T, .) saved-state tensors and into the
 * staging rows of the next GEMM.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
  int B, H;
  const float* z;         long long ldz;        /* (B, >=4H) gate pre-activations, order i,f,g,o (:777-783) */
  const float* c_prev;    long long ld_cprev;   /* (B,H) */
  const float* gate_pre;  long long ld_gate_pre;/* optional (B,H): x_gate(x) + h_gate(h_old), :982          */
  float *h, *c;           long long ld_state;   /* new state rows                                           */
  float *g, *i, *f, *s;   long long ld_gate;    /* pre-tanh candidate, input/forget gates, sentinel (if gate_pre) */
  float* h_copy0;         long long ld_copy0;   /* optional copies of h (inputs of the next GEMMs)          */
  float* h_copy1;         long long ld_copy1;
  float* h_copy2;         long long ld_copy2;
  float* s_copy;          long long ld_s_copy;
  float *o, *sg;                                /* optional (stride ld_gate): sigmoid(output gate), sigmoid(sentinel gate) —
                                                   the saved state of the gradient explainers, gridTDmodel.py:1381,1409 */
} lrpx_lstm_cell_args;

int lrpx_lstm_cell_f32(const lrpx_lstm_cell_args* args, void* stream);

/* One LSTM time step as ONE kernel: skinny fp32 GEMM (B <= a few hundred rows) + the cell update of
 * lrpx_lstm_cell_f32 in its epilogue.     z[b][g*H + j] = add[b][g*H + j] + sum_k x[b][k] * W[k][g*H + j]
 * G = 4 (gates i,f,g,o) or 5 (+ the sentinel gate pre-activation, gridTDmodel.py:982).  Each CTA owns 4 hidden
 * units with all their G gate columns, so the cell update needs no second pass.  `wp` is W re-laid out once by
 * lrpx_lstm_prep_weights_f32 as [H/4][G][4][K] (each CTA's 4*G weight rows contiguous, k fastest). */
int lrpx_lstm_prep_weights_f32(const float* w /* (K, G*H) row-major */, float* wp, int K, int G, int H, void* stream);

typedef struct {
  int B, H, K, G;
  const float* x;         long long ldx;        /* (B,K) concatenated recurrent inputs                       */
  const float* wp;                              /* prepared weights                                          */
  const float* add;       long long ld_add;     /* (B,G*H) addend rows, or one (G*H) row with ld_add = 0     */
  const float* c_prev;    long long ld_cprev;
  float *h, *c;           long long ld_state;
  float *g, *i, *f, *s;   long long ld_gate;    /* s: sentinel, required when G == 5                         */
  float* h_copy0;         long long ld_copy0;
  float* h_copy1;         long long ld_copy1;
  float* h_copy2;         long long ld_copy2;
  float* s_copy;          long long ld_s_copy;
  float *o, *sg;                                /* optional, as in lrpx_lstm_cell_args                       */
} lrpx_lstm_step_args;

int lrpx_lstm_step_f32(const lrpx_lstm_step_args* args, void* stream);

/* AdaptiveAttention.forward (gridTDmodel.py:61-103), one block per image:
 *   z[p] = w_h . tanh(img_proj[b,p,:] + hproj[b,p]) (sic, needs P == K);  alpha = softmax z;  ctx = sum_p alpha[p] A[b,p,:]
 *   zs = w_h . tanh(sproj[b,:] + hproj[b,:]);  beta = softmax([z; zs])[-1];  ctx_hat = beta*s + (1-beta)*ctx */
typedef struct {
  int B, P, K, H;                              /* K = n_pixel of the attention projections */
  const float* A;                              /* (B,P,H) projected features, pixel-major  */
  const float* img_proj;                       /* (B,P,K) W_v_proj(A)                      */
  const float* hs_proj;   long long ld_hs;     /* (B,2K): [W_g_proj(h) | W_s_proj(s)+bias], or NULL: computed in the
                                                  kernel from h, s and the projection weights below            */
  const float* w_h;                            /* (K)                                      */
  const float* s;         long long ld_s;      /* (B,H) sentinel                           */
  float *ctx, *ctx_hat;   long long ld_out;
  float* alpha;           long long ld_alpha;  /* (B,P) rows */
  float* beta;            long long ld_beta;   /* (B) */
  float* ctx_hat_copy;    long long ld_copy;   /* optional */
  const float* h;         long long ld_h;      /* (B,H) hidden state (hs_proj == NULL)      */
  const float *W_g, *W_s, *b_s;                /* (K,H), (K,H), (K) projection weights      */
} lrpx_ada_attention_args;

int lrpx_adaptive_attention_f32(const lrpx_ada_attention_args* args, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core path (tcgen05 + TMA, bf16 operands / fp32 accumulate in TMEM).
 *
 * Layout "PF" (padded-flat NHWC bf16): an image of h x w pixels and C channels is a block of
 * (h+1)*(w+1) pixel rows of C bf16; block row 0 and block column 0 are zero padding and pixel (y,x) sits
 * at block offset (y+1)*(w+1)+(x+1).  The right/bottom halo of one image is the left/top padding of what
 * follows, so the 3x3 neighbour (dy,dx) of flat row p is row p + dy*(w+1) + dx and a 3x3/stride-1/pad-1
 * convolution is 9 accumulated GEMMs over row-shifted views of one 2-D (rows x channels) tensor.
 *
 * One implicit-GEMM kernel family serves the activation-producing forward (+ z+), and the relevance
 * (transposed-conv) pass:      acc[p][n] = sum_{tap,c} A[p + off(tap)][c] * Wt[n][tap*cin + c]
 *
 * Relevance chain (alpha=1, beta=0; LRPtools/lrp_modules.py:81-84,134, LRPtools/utils.py:16-31): with
 * gain_l = a_{l+1} / safe(z+_l) (per image, independent of the explained word) the per-explanation work of
 * one conv layer is ONE contraction   s_{l-1} = gain_{l-1} (.) (W+_l^T * s_l),   s_l = R_{l+1}/safe(z+_l).
 * ------------------------------------------------------------------------------------------- */
enum {
  /* dual tile: Wt holds, per tile of `half` output channels, the W rows then the W+ rows (ncol = 2*cout):
   *   act[p][n]  = relu(acc_w + bias[n])                                (forward, lrp_wrapper.py:70)
   *   gain[p][n] = act[p][n] / safe(acc_w+)   (gain_mode 0)   or   1 / safe(acc_w+)   (gain_mode 1)
   *   safe(z) = z + 1e-7*[z==0]                                          (utils.py:16-18)
   * out = act (PF bf16), out2 = gain (PF bf16); padding rows are written as zeros. */
  LRPX_TC_EPI_FWD_GAIN = 1,
  /* out[p][n] = bf16(acc[p][n] * gain[img(p)][rem(p)][n]); padding rows -> 0
   *   (R_in = a (.) c, then the division by z+ of the layer below: lrp_modules.py:134, utils.py:26-30) */
  LRPX_TC_EPI_MUL = 2,
  /* as MUL but the tile is at pooled resolution (h, w = pooled size): `gain` and `pool_idx` are pooled-size
   * PF tensors, pool_idx holds the argmax 0..3 (dy*2+dx) of each 2x2 window; every pooled pixel writes its
   * 4 fine pixels in the (2h x 2w) PF output, the product at the winner and 0 elsewhere
   *   (max-pool winner-take-all, lrp_modules.py:186-191) */
  LRPX_TC_EPI_MUL_UNPOOL = 3,
  /* first layer: ncol = 16, acc columns 0..2 = W+^T s, 3..5 = W-^T s;
   *   out_f32[e][c][y][x] (NCHW, unpadded) = max(x,0)*acc[c] + min(x,0)*acc[3+c]   (lrp_modules.py:81-84) */
  LRPX_TC_EPI_INPUT = 4,
  /* out_f32[p][n] = acc[p][n] (debug / tests of the GEMM machinery) */
  LRPX_TC_EPI_STORE_F32 = 5,
  /* decoder projector rule (gridTDmodel.py:1121-1128, aoamodel.py:1141-1150), blocks = requests, rows = pixels:
   *   out_f32[q][p][n] = x[img(q)][p][n] * (acc[q*P+p][n] + bias[q][n])
   * x = fp32 (n_x, P, ncol) encoder features, bias = fp32 (n_img, ncol) per-request addend or NULL */
  LRPX_TC_EPI_FEAT = 6,
  /* as FEAT, divided by stab(x1[img(q)][p][n])  (z + 0.01*sign z, 0 -> 0.01; the value-projection rule) */
  LRPX_TC_EPI_FEAT_DIV = 7,
  /* first layer with the three filter columns folded into N: ncol = 24, Wt row dx*8 + c (c = 0..2: W+^T, 3..5: W-^T,
   * 6..7: zero) holds, K-ordered (filter row dy, channel), the weights of filter tap (dy, dx); the kernel adds the
   * three column-shifted partial sums in its epilogue.  Same output as LRPX_TC_EPI_INPUT (3x3 only).
   * gain_mode selects the delivery format of the heat-map: 0 = fp32 (n, 3, h, w), 1 = channel mean fp32 (n, h, w)
   * (evaluation.py:134,411,503 reduce every heat-map with torch.mean(relevance, dim=(0,1)) first), 2 = fp16 (n, 3, h, w).
   * With cam_rows set (guided rule only) every pixel's three values are first multiplied by Guided Grad-CAM's expanded map
   *   v[e][y][x] = sum_j cam_kw[x][j] * cam_rows[e][y][j]   (fmaf over j = 0..cam_w-1, lrpx_cam_expand_mul_f32's order)
   * so format 0 equals lrpx_cam_expand_mul_f32 of the un-multiplied output bit for bit, and 1 / 2 are its formats. */
  LRPX_TC_EPI_INPUT3 = 8,
  /* General relevance epilogue (any alpha/beta, the epsilon rule, bf16 or fp32-accurate storage):
   *   for group j < groups:  v_j = acc[p][n] * gain_j[img(p)][rem(p)][n]
   *   split == 0: out[p][j*ncol + n] = bf16(v_j)                      gains are bf16 PF (rows, ncol)
   *   split == 1: out[p][j*ncol + n] = hi(v_j), out[p][(groups+j)*ncol + n] = lo(v_j) with v = hi + lo, both bf16
   *               (16 significant bits); gains are fp32 PF (rows, ncol)
   * The row written is the A operand of the layer below: groups = 2 carries [alpha*R/z+ | -beta*R/z-] so that
   * alpha*R(pos-net) - beta*R(neg-net) (lrp_modules.py:129-150) is ONE contraction over K = [W+^T | W-^T]. */
  LRPX_TC_EPI_MULX = 9,
  /* MULX at pooled resolution with the max-pool winner-take-all scatter of MUL_UNPOOL */
  LRPX_TC_EPI_MULX_UNPOOL = 10,
  /* General forward + gains.  Wt holds per tile of `half` output channels n_acc row blocks: W, then W+ (n_acc >= 2),
   * then W- (n_acc == 3);  z = acc_W + bias, act = relu(z);  num = act (gain_mode 0) or 1 (gain_mode 1)
   *   rule 0 (alpha-beta): gain0 = alpha * num / safe(acc_W+ [+ bias if zbias]),
   *                        gain1 = -beta * num / safe(acc_W- [+ bias if zbias])                      (n_acc == 3)
   *   rule 1 (epsilon, lrp_modules.py:9-24 on the unfolded conv): gain0 = num' / stab(acc_W [+ bias if zbias]),
   *                        num' = num with exact zeros replaced by -1e-6 (Q9), stab(z) = z + 0.01 sign z, 0 -> 0.01
   *   rule 2 (gradient, gridTDmodel.py:1510-1523) / 3 (guided backpropagation, :1677-1723): n_acc == 1,
   *                        gain0 = [act > 0], the ReLU's derivative.  With rule 3 the MULX epilogues pass only the positive
   *                        part of the accumulator (the ReLU backward hook of :1680-1686); with rule >= 2 INPUT3 returns
   *                        W^T g itself (rows 0..2 of its weight), not multiplied by the image.
   * out = act (bf16 PF, or hi|lo split with 2*cout channels per row when split), out2 = gain0, out3 = gain1
   * (bf16, or fp32 when split). */
  LRPX_TC_EPI_FWDX = 11,
};

/* lrpx_tc_conv_args.fwd_flags bit for LRPX_TC_EPI_MUL with ncol == 64 (3x3): the three filter COLUMNS are folded into
 * the GEMM's N — Wt holds 3 * ncol rows, row dx * ncol + n, K ordered (filter row, channel), 3 * cin columns — and the
 * epilogue adds the three column-shifted partial sums.  A 64-column MMA is bound by its shared-memory operand reads;
 * the folded form does a third of the MMAs at three times the width.  Same result up to the fp32 summation order. */
#define LRPX_TC_FOLD_COLUMNS 8

typedef struct {
  int n_img;            /* PF blocks in A (images or explanations)                                */
  int h, w;             /* unpadded spatial size of A's blocks (== output size)                   */
  int cin;              /* channels of A (multiple of 64)                                         */
  int ncol;             /* rows of Wt == GEMM N                                                   */
  int ksize;            /* 1 or 3                                                                 */
  int epilogue;         /* LRPX_TC_EPI_*                                                          */
  int gain_mode;        /* FWD_GAIN / FWDX: 0 act/z, 1 1/z;  INPUT3: delivery format (see above)   */
  const void* a;        /* bf16 PF (n_img, (h+1)*(w+1), cin)                                      */
  const void* wt;       /* bf16 (ncol, ksize*ksize*cin), K ordered (tap, channel)                 */
  const float* bias;    /* FWD_GAIN: (cout) or NULL                                               */
  const void* gain;     /* bf16 PF (n_gain_img, blk, ncol), MUL / MUL_UNPOOL                      */
  const int32_t* row_img; /* (n_img) block of `gain`/`pool_idx`/`x` used by each block of A; NULL = identity */
  const uint8_t* pool_idx;/* PF (n_gain_img, blk, ncol) argmax bytes, MUL_UNPOOL                  */
  const float* x;       /* fp32 NCHW (n_x, 3, h, w) input images, INPUT; fp32 (n_x, blk, ncol), FEAT  */
  void* out;
  void* out2;
  const float* x1;      /* FEAT_DIV: fp32 (n_x, blk, ncol)                                        */
  /* ---- general modes (MULX / MULX_UNPOOL / FWDX; zero for the epilogues above) */
  const void* gain2;    /* MULX*: gain of group 1                                                 */
  void* out3;           /* FWDX: gain of group 1                                                  */
  int a_phys;           /* channels per row of A in memory when they differ from `cin` (0 = cin): with
                         * a_phys < cin the K blocks beyond a_phys wrap around (block kc reads A block
                         * kc - a_phys/64), so a hi|lo split row [hi | lo] serves the error-compensated
                         * product a*w ~ hi*w_hi + lo*w_hi + hi*w_lo as K = [hi | lo | hi] x [w_hi | w_hi | w_lo]
                         * without storing hi twice                                                */
  int groups;           /* MULX*: 1 or 2 gain groups                                              */
  int split;            /* 0: bf16 rows / bf16 gains; 1: hi|lo split rows / fp32 gains            */
  int n_acc;            /* FWDX: 1, 2 or 3 accumulators per output channel                        */
  int rule;             /* FWDX: 0 alpha-beta, 1 epsilon                                          */
  int zbias;            /* FWDX: the bias enters the rule's divisor (ignore_bias = False)         */
  float alpha, beta;    /* FWDX                                                                   */
  /* ---- residual networks (models/resnet.py:95-140, lrp_modules.py:197-280) */
  const void* add;      /* MULX: per-block addend rows (bf16, `add_pitch` elements per row): the relevance of the other
                         * branch at a fork;  out_j = acc * gain_j + add * gainB_j   (gainB_0 = gain3, gainB_1 = gain4).
                         * With out2 set and two groups the groups go to two separate (rows, ncol) bf16 tensors
                         * (out, out2) instead of one K-concatenated row.
                         * MULX_UNPOOL with pool_idx == NULL writes every product at the FIRST pixel of its 2x2 block:
                         * the zero-stuffing of a stride-2 transposed convolution.                              */
  const void* gain3;
  const void* gain4;
  const float* bn_w;    /* FWDX: folded BatchNorm y = z*bn_w[n] + bn_b[n] (eval mode) and its rule
                         * R = |z w| / (|z w| + |b|) R_out (lrp_modules.py:204-215) as a factor of gain0           */
  const float* bn_b;
  const void* idn;      /* FWDX: identity branch (bf16 PF, cout channels; hi|lo rows of 2*cout when split): out = relu(y + idn),
                         * Add rule ratios rho1 = y / stab'(y+idn) (factor of gain0), rho2 = idn / stab'(y+idn); out3 = rho2 * hd */
  const void* hd;       /* FWDX: PF factor of the identity-branch gain (the downsample conv's ratio / z+; bf16, fp32 when
                         * split) or NULL */
  void* out4;           /* FWDX: act * gain0                                                       */
  void* out5;           /* FWDX: act * out3                                                        */
  int add_pitch;
  int fwd_flags;        /* FWDX: bit 0 = no ReLU (downsample branch), bit 1 = keep the even pixels only and store
                         * them into a PF tensor of half the resolution (stride-2 convolution);
                         * STORE_F32: bit 2 = store bf16 (rows of ncol bf16) instead of fp32              */
  int out_pitch;        /* STORE_F32: floats per row of `out` (0 = ncol) and                                */
  int n_valid;          /*            the columns that exist (<= ncol; the weight rows beyond are padding);
                         *            `bias` (n_valid floats) is added when given                           */
  /* ---- Guided Grad-CAM factor of INPUT3 with rule 3 (NULL cam_rows: no factor) */
  const float* cam_rows;  /* fp32 (n_img, h, cam_w): lrpx_cam_expand_rows_f32 of each block's Grad-CAM map       */
  const float* cam_kw;    /* fp32 (w, cam_w): the expansion along x (the Kw of lrpx_cam_expand_mul_f32)          */
  int cam_w;              /* width of the Grad-CAM map, 1..64                                                    */
} lrpx_tc_conv_args;

int lrpx_tc_conv(const lrpx_tc_conv_args* args, void* stream);

/* Plain tensor-core GEMM of the same kernel family (one filter tap):  out[m][n] = sum_k a[m][k] * wt[n][k]
 *   a (m,k) bf16 row-major, wt (n,k) bf16 row-major, out (m,n) fp32.  k % 64 == 0, n % 32 == 0, n <= 256 or n % 256 == 0.
 * Used by the decoder kernels for their error-compensated bf16x3 GEMMs (LRPX_DEC_TC_GEMM). */
int lrpx_tc_gemm_bf16_f32(const void* a, const void* wt, float* out, int m, int n, int k, void* stream);

/* Linear layer / GEMM at fp32 accuracy on the tensor cores (error-compensated bf16x3, see a_phys above):
 *   out[m][n] = sum_k a[m][k] * W[n][k] + bias[n]         a fp32 (m, k) with row pitch lda, out fp32 with row pitch ldo
 * w3 = the prepared weight: bf16 (n_pad, 3k) rows [hi | hi | lo] of W, n_pad >= n a multiple of 32 (<= 256) or of 256, rows
 * beyond n zero.  k % 64 == 0, n % 4 == 0, ldo % 4 == 0.  workspace: lrpx_gemm_x3_workspace_bytes(m, k) bytes (the hi | lo
 * split of a).  Replaces the library GEMMs of the explainer forward (gridTDmodel.py:941-1012: projector, attention
 * projections, gate pre-activations, vocabulary projection). */
size_t lrpx_gemm_x3_workspace_bytes(int m, int k);
int lrpx_gemm_x3_f32(const float* a, int lda, const void* w3, int n_pad, const float* bias, float* out, int ldo, int m, int n,
                     int k, void* workspace, size_t workspace_bytes, void* stream);

/* First VGG layer forward on CUDA cores (cin = 3 is no tensor-core shape): from fp32 NCHW images
 *   act  = relu(conv(x, W) + b)                       -> PF bf16 (n, blk, cout)
 *   gain = act / safe(conv(x+, W+) + conv(x-, W-))    -> PF bf16                  (lrp_modules.py:81-84)
 * cout must be a multiple of 8; 3x3, stride 1, pad 1. */
int lrpx_tc_first_fwd(const float* x, const float* w, const float* bias, void* act, void* gain, int n, int h, int wd,
                      int cout, void* stream);

/* First VGG layer on the tensor cores: sign-split im2col of the fp32 NCHW images (n,3,h,w) into PF bf16 rows of 64
 * columns [x+ over the 27 (ci,r,s) taps | x- over the 27 taps | 10 zeros].  lrpx_tc_conv(ksize 1, cin 64,
 * LRPX_TC_EPI_FWD_GAIN) with weight rows [w | w | 0] (z) and [w+ | w- | 0] (z+) then yields act and gain of
 * the mixed-sign first layer (lrp_modules.py:81-84). */
int lrpx_tc_im2col3_split_bf16(const float* x, void* dst, int n, int h, int w, void* stream);

/* One-time weight preparation (replaces the per-call PosNetConv/NegNetConv clones,
 * lrp_modules.py:59-76): from fp32 (cout,cin,kh,kw) build bf16 GEMM operands.
 *   mode 0: forward      Wt[co][(r,s,ci)]            = W[co][ci][r][s]
 *   mode 1: forward W+   Wt[co][(r,s,ci)]            = max(W,0)
 *   mode 2: relevance    Wt[ci][(r,s,co)]            = max(W[co][ci][kh-1-r][kw-1-s],0)   (transposed conv)
 *   mode 3: relevance W- Wt[ci][(r,s,co)]            = min(W[co][ci][kh-1-r][kw-1-s],0)
 * rows/cols beyond the source are zero-filled up to (rows_pad, chan_pad) so tiles never read junk. */
int lrpx_weight_prep_bf16(const float* w, void* wt, int cout, int cin, int kh, int kw, int mode, int rows_pad,
                          int chan_pad, void* stream);

/* 2x2/2 max-pool on PF bf16 with argmax (0..3 = dy*2+dx, PyTorch scan order: first maximum wins, NaN wins)
 * and the gain gathered at the winner:  pooled[p][c] = max, idx[p][c], gain_pooled[p][c] = gain_fine[winner][c].
 * (h, w) is the fine size (even).  gain_fine/gain_pooled may both be NULL; idx may be NULL. */
int lrpx_tc_maxpool2_bf16(const void* act, const void* gain_fine, void* pooled, uint8_t* idx, void* gain_pooled,
                          int n, int h, int w, int c, void* stream);
/* entry of the relevance chain:  s_top[e][pf(p)][c] = bf16( r[e][p][c] * rz[row_img[e]][pf(p)][c] ),
 * r is fp32 pixel-major (n_expl, h*w, c) as produced by the decoder kernels; padding rows -> 0 */
int lrpx_tc_scale_rows(const float* r, const void* rz, const int32_t* row_img, void* out, int n_expl, int h, int w,
                       int c, void* stream);
/* PF bf16 (n, blk, c) -> dense fp32: layout 0 = pixel-major (n, h*w, c), 1 = NCHW (n, c, h, w) */
int lrpx_tc_pf_to_dense_f32(const void* src, float* dst, int n, int h, int w, int c, int layout, void* stream);
/* dense fp32 NCHW (n, c, h, w) -> PF bf16 (n, blk, c_pad), channels >= c zero-filled */
int lrpx_tc_nchw_to_pf_bf16(const float* src, void* dst, int n, int c, int h, int w, int c_pad, void* stream);

/* ---- companions of the general modes (groups = 1 | 2 gain groups; split = 0: bf16, 1: hi|lo rows + fp32 gains) */
/* lrpx_tc_im2col3_split_bf16 with hi|lo rows: 128 columns [hi of the 64 | lo of the 64] */
int lrpx_tc_im2col3_split_x(const float* x, void* dst, int n, int h, int w, int split, void* stream);
/* lrpx_tc_maxpool2_bf16 for split rows (the winner is the largest hi+lo) and up to two gain tensors */
int lrpx_tc_maxpool2_x(const void* act, const void* gain0_fine, const void* gain1_fine, void* pooled, uint8_t* idx,
                       void* gain0_pooled, void* gain1_pooled, int n, int h, int w, int c, int split, void* stream);
/* lrpx_tc_scale_rows for the general chain: out row = [r*rz0 | r*rz1] (groups), bf16 or hi|lo split.
 * split bit 1 (value 2): r is clamped at 0 first — the entry of guided backpropagation (gridTDmodel.py:1680-1686) */
int lrpx_tc_scale_rows_x(const float* r, const void* rz0, const void* rz1, const int32_t* row_img, void* out,
                         int n_expl, int h, int w, int c, int groups, int split, void* stream);
/* ---- residual-network encoder (models/resnet.py:143-239): stem and strides, bf16 PF */
/* conv1 (7x7 / stride 2 / pad 3, mixed-sign input): sign-split im2col at the output resolution (h/2, w/2): rows of 320
 * bf16 [x+ over the 147 (ci,ky,kx) taps | x- over the 147 taps | 26 zeros] for lrpx_tc_conv(ksize 1, cin 320, FWDX). */
int lrpx_tc_im2col7s2_split_bf16(const float* x, void* dst, int n, int h, int w, void* stream);
/* 3x3 / stride 2 / pad 1 max-pool of a post-ReLU PF tensor (h, w even): pooled (h/2, w/2) and idx = ky*3+kx of the winner
 * (PyTorch scan order, first maximum wins), 255 where the maximum is 0 (no relevance passes, lrp_modules.py:186-191). */
int lrpx_tc_maxpool3s2_bf16(const void* act, void* pooled, uint8_t* idx, int n, int h, int w, int c, void* stream);
/* relevance through that pool, gather form over the overlapping windows, times the per-image gain of the layer below:
 * out[e][i][j][c] = gain[row_img[e]][i][j][c] * sum_{windows (y,x) containing (i,j) with winner (i,j)} r[e][y][x][c] */
int lrpx_tc_unpool3s2_bf16(const void* r, const uint8_t* idx, const void* gain, const int32_t* row_img, void* out, int n_expl,
                           int h, int w, int c, void* stream);
/* dst (n, h/2, w/2) <- src (n, h, w) at the even pixels (input of a 1x1 / stride 2 convolution) */
int lrpx_tc_subsample2_bf16(const void* src, void* dst, int n, int h, int w, int c, void* stream);
/* stem relevance: gathers the image relevance from P (n_expl * (h/2+1)*(w/2+1) rows of ldp floats, column
 * (ky*7+kx)*6 + s*3 + c = sum_ch A[q][ch] W(s)[ch][c][ky][kx], s = 0: W+, 1: W-) written by the 1x1 GEMM
 * (lrpx_tc_conv, STORE_F32):  heat = x+ * sum P[..][0][c] + x- * sum P[..][1][c];  mode as LRPX_TC_EPI_INPUT3's. */
int lrpx_tc_stem_col2im_f32(const float* P, int ldp, const float* x, const int32_t* row_img, void* out, int n_expl, int h,
                            int w, int mode, void* stream);
/* the same with P stored as bf16 (lrpx_tc_conv STORE_F32 with fwd_flags bit 2): half the bytes of the intermediate */
int lrpx_tc_stem_col2im_bf16(const void* P, int ldp, const float* x, const int32_t* row_img, void* out, int n_expl, int h,
                             int w, int mode, void* stream);
/* lrpx_tc_pf_to_dense_f32 for hi|lo rows of 2*c channels (value = hi + lo) */
int lrpx_tc_pf_split_to_dense_f32(const void* src, float* dst, int n, int h, int w, int c, int layout, void* stream);
/* ---- the residual-network stem in the fp32-accurate forward (split = 0: exactly the bf16 functions above) */
/* lrpx_tc_im2col7s2_split_bf16 with hi|lo rows (split = 1): 640 bf16 [hi of the 320 | lo of the 320], hi + lo ~ the fp32
 * tap; hi is the bf16 function's row.  The A operand of lrpx_tc_conv(ksize 1, cin 960, a_phys 640, split 1, FWDX) with
 * weight rows [hi | hi | lo] of [w | w | 0] and [w+ | w- | 0] (models/resnet.py:143-149, lrp_modules.py:81-84). */
int lrpx_tc_im2col7s2_split_x(const float* x, void* dst, int n, int h, int w, int split, void* stream);
/* lrpx_tc_maxpool3s2_bf16 on hi|lo rows (split = 1, 2*c bf16 per row): the winner is the largest hi + lo, first maximum in
 * PyTorch scan order, idx = 255 where the maximum is 0; pooled keeps the winner's hi|lo row (resnet.py:150,
 * lrp_modules.py:186-191).  lrpx_tc_subsample2_bf16 with c = 2*c serves hi|lo rows as they are. */
int lrpx_tc_maxpool3s2_x(const void* act, void* pooled, uint8_t* idx, int n, int h, int w, int c, int split, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* LRPX_H_ */
