"""ctypes binding of liblrpx.so (include/lrpx.h).  The product path has NO CPU fallback: if the
library is missing or a call fails, an exception is raised."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "liblrpx.so")


class LrpxError(RuntimeError):
    pass


class ConvShape(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "cin", "h", "w", "cout", "kh", "kw", "stride_h", "stride_w", "pad_h",
                                       "pad_w", "dil_h", "dil_w")]


class PoolShape(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n", "c", "h", "w", "kh", "kw", "stride_h", "stride_w", "pad_h", "pad_w")]


_P = C.c_void_p
_GRID_PTRS = ["feat", "avg", "A_pre", "A", "glob_pre", "x1", "x2", "h1", "c1", "h2", "c2", "g1", "i1", "f1", "g2",
              "i2", "f2", "st", "ctx", "ctx_hat", "alpha", "beta", "pred", "W_g1", "W_g2", "W_fc", "W_glob", "W_proj",
              "req_img", "req_t", "req_word", "r_feat", "r_words", "r_words_raw"]


class GridTDArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "T", "H", "E", "P", "C", "V", "Q", "flags", "reserved_")] + \
               [(n, _P) for n in _GRID_PTRS]


_AOA_PTRS = ["feat", "A_pre", "A", "glob", "value", "x", "h", "c", "g", "i", "ctx", "caoa", "caoa_lin", "alpha",
             "pred", "W_g", "W_fc", "W_aoa", "W_v", "W_proj", "req_img", "req_t", "req_word", "req_head", "r_feat",
             "r_words", "r_words_raw"]


class AoaArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "T", "H", "E", "P", "C", "V", "Q", "num_head", "flags")] + \
               [(n, _P) for n in _AOA_PTRS]


_GRID_GRAD_PTRS = ["feat", "c1", "c2", "g1", "i1", "f1", "o1", "g2", "i2", "f2", "o2", "sg", "alpha", "beta", "W1", "W2",
                   "W_fc", "W_glob", "W_proj", "req_img", "req_t", "req_word", "d_feat", "r_words", "r_words_raw"]


class GridTDGradArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "T", "H", "E", "P", "C", "V", "Q", "flags", "reserved_")] + \
               [(n, _P) for n in _GRID_GRAD_PTRS]


_AOA_GRAD_PTRS = ["c", "g", "i", "f", "o", "caoa_gate", "caoa_lin", "alpha", "W_g", "W_fc", "W_aoa", "W_gate", "W_v",
                  "W_proj", "req_img", "req_t", "req_word", "req_head", "d_feat", "r_words", "r_words_raw"]


class AoaGradArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "T", "H", "E", "P", "C", "V", "Q", "num_head", "flags")] + \
               [(n, _P) for n in _AOA_GRAD_PTRS]


_ADA_GRAD_PTRS = ["c", "g", "i", "f", "o", "sg", "alpha", "beta", "W_g", "W_fc", "W_glob", "W_proj", "req_img", "req_t",
                  "req_word", "d_feat", "r_words", "r_words_raw"]


class AdaptiveGradArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "T", "H", "E", "P", "C", "V", "Q", "flags", "reserved_")] + \
               [(n, _P) for n in _ADA_GRAD_PTRS]


_ADA_PTRS = ["feat", "avg", "z_proj", "A", "z_glob", "x", "h", "c", "g", "i", "f", "st", "ctx", "ctx_hat", "alpha", "beta",
             "pred", "W_g", "W_fc", "W_glob", "W_proj", "req_img", "req_t", "req_word", "r_feat", "r_words",
             "r_words_raw"]


class AdaptiveArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "T", "H", "E", "P", "C", "V", "Q", "flags", "reserved_")] + \
               [(n, _P) for n in _ADA_PTRS]


class TcConvArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("n_img", "h", "w", "cin", "ncol", "ksize", "epilogue", "gain_mode")] + \
               [(n, _P) for n in ("a", "wt", "bias", "gain", "row_img", "pool_idx", "x", "out", "out2", "x1", "gain2",
                                  "out3")] + \
               [(n, C.c_int) for n in ("a_phys", "groups", "split", "n_acc", "rule", "zbias")] + \
               [("alpha", C.c_float), ("beta", C.c_float)] + \
               [(n, _P) for n in ("add", "gain3", "gain4", "bn_w", "bn_b", "idn", "hd", "out4", "out5")] + \
               [("add_pitch", C.c_int), ("fwd_flags", C.c_int), ("out_pitch", C.c_int), ("n_valid", C.c_int)] + \
               [("cam_rows", _P), ("cam_kw", _P), ("cam_w", C.c_int)]


_LL = C.c_longlong


class LstmCellArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("H", C.c_int), ("z", _P), ("ldz", _LL), ("c_prev", _P), ("ld_cprev", _LL),
                ("gate_pre", _P), ("ld_gate_pre", _LL), ("h", _P), ("c", _P), ("ld_state", _LL), ("g", _P), ("i", _P),
                ("f", _P), ("s", _P), ("ld_gate", _LL), ("h_copy0", _P), ("ld_copy0", _LL), ("h_copy1", _P),
                ("ld_copy1", _LL), ("h_copy2", _P), ("ld_copy2", _LL), ("s_copy", _P), ("ld_s_copy", _LL),
                ("o", _P), ("sg", _P)]


class LstmStepArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("H", C.c_int), ("K", C.c_int), ("G", C.c_int), ("x", _P), ("ldx", _LL), ("wp", _P),
                ("add", _P), ("ld_add", _LL), ("c_prev", _P), ("ld_cprev", _LL), ("h", _P), ("c", _P),
                ("ld_state", _LL), ("g", _P), ("i", _P), ("f", _P), ("s", _P), ("ld_gate", _LL), ("h_copy0", _P),
                ("ld_copy0", _LL), ("h_copy1", _P), ("ld_copy1", _LL), ("h_copy2", _P), ("ld_copy2", _LL),
                ("s_copy", _P), ("ld_s_copy", _LL), ("o", _P), ("sg", _P)]


class AdaAttentionArgs(C.Structure):
    _fields_ = [("B", C.c_int), ("P", C.c_int), ("K", C.c_int), ("H", C.c_int), ("A", _P), ("img_proj", _P),
                ("hs_proj", _P), ("ld_hs", _LL), ("w_h", _P), ("s", _P), ("ld_s", _LL), ("ctx", _P), ("ctx_hat", _P),
                ("ld_out", _LL), ("alpha", _P), ("ld_alpha", _LL), ("beta", _P), ("ld_beta", _LL),
                ("ctx_hat_copy", _P), ("ld_copy", _LL), ("h", _P), ("ld_h", _LL), ("W_g", _P), ("W_s", _P), ("b_s", _P)]


class BeamArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("B", "k", "V", "L", "step", "end_id")] + \
               [(n, _P) for n in ("logits", "scores", "n_alive", "seqs", "comp_seqs", "comp_len", "comp_scores", "n_comp",
                                  "prev_words", "src_row")]


BEAM_GATHER_MAX = 8


class BeamGatherArgs(C.Structure):
    _fields_ = [("n_rows", C.c_int), ("n_pairs", C.c_int), ("src_row", _P), ("dst", _P * BEAM_GATHER_MAX),
                ("src", _P * BEAM_GATHER_MAX), ("ld_dst", _LL * BEAM_GATHER_MAX), ("ld_src", _LL * BEAM_GATHER_MAX),
                ("width", C.c_int * BEAM_GATHER_MAX)]


class BlockImageArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("Q", "C", "H", "W", "patch", "k", "img_c", "reserved_")] + \
               [(n, _P) for n in ("heat", "images", "req_img", "mask", "masked")]


class BboxArgs(C.Structure):
    _fields_ = [(n, C.c_int) for n in ("Q", "C", "H", "W", "n_thr", "max_boxes")] + [("sign", C.c_float), ("inplace_quirk", C.c_int)] + \
               [(n, _P) for n in ("heat", "thresholds", "boxes", "n_boxes", "ratio")]


# every symbol include/lrpx.h declares: name -> (restype, argtypes)
_i, _f, _sz = C.c_int, C.c_float, C.c_size_t
SYMBOLS = {
    "lrpx_last_error": (C.c_char_p, []),
    "lrpx_version": (_i, []),
    "lrpx_device_cc": (_i, []),
    "lrpx_conv_rule_s_f32": (_i, [_P, _P, _P, _P, _P, _P, C.POINTER(ConvShape), _i, _P]),
    "lrpx_conv_rule_rin_f32": (_i, [_P, _P, _P, _P, C.POINTER(ConvShape), _i, _f, _i, _P]),
    "lrpx_conv_forward_f32": (_i, [_P, _P, _P, _P, C.POINTER(ConvShape), _i, _P]),
    "lrpx_linear_eps_f32": (_i, [_P, _P, _P, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_maxpool_forward_f32": (_i, [_P, _P, _P, C.POINTER(PoolShape), _P]),
    "lrpx_maxpool_wta_f32": (_i, [_P, _P, _P, C.POINTER(PoolShape), _P]),
    "lrpx_avgpool_prop_f32": (_i, [_P, _P, _P, C.POINTER(PoolShape), _P]),
    "lrpx_bn_absratio_f32": (_i, [_P, _P, _P, _P, _P, _P, _P, _f, _i, _i, _i, _P]),
    "lrpx_add_split_f32": (_i, [_P, _P, _P, _P, _P, _sz, _P]),
    "lrpx_relu_mask_f32": (_i, [_P, _P, _P, _sz, _P]),
    "lrpx_normalize_relevance_f32": (_i, [_P, _P, _i, _i, _f, _P]),
    "lrpx_sum_f64": (_i, [_P, _sz, _P, _P]),
    "lrpx_lrp_linear_eps_workspace_bytes": (_sz, [_i, _i]),
    "lrpx_lrp_linear_eps_f32": (_i, [_P, _P, _P, _P, _P, _i, _i, _P, _sz, _P]),
    "lrpx_lrp_mha_f32": (_i, [_P, _P, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_gridtd_decoder_workspace_bytes": (_sz, [C.POINTER(GridTDArgs)]),
    "lrpx_gridtd_decoder_lrp_f32": (_i, [C.POINTER(GridTDArgs), _P, _sz, _P]),
    "lrpx_gridtd_decoder_grad_workspace_bytes": (_sz, [C.POINTER(GridTDGradArgs)]),
    "lrpx_gridtd_decoder_grad_f32": (_i, [C.POINTER(GridTDGradArgs), _P, _sz, _P]),
    "lrpx_aoa_decoder_grad_workspace_bytes": (_sz, [C.POINTER(AoaGradArgs)]),
    "lrpx_aoa_decoder_grad_f32": (_i, [C.POINTER(AoaGradArgs), _P, _sz, _P]),
    "lrpx_adaptive_decoder_grad_workspace_bytes": (_sz, [C.POINTER(AdaptiveGradArgs)]),
    "lrpx_adaptive_decoder_grad_f32": (_i, [C.POINTER(AdaptiveGradArgs), _P, _sz, _P]),
    "lrpx_grad_cam_f32": (_i, [_P, _P, _P, _P, _i, _i, _i, _P]),
    "lrpx_cam_expand_mul_f32": (_i, [_P, _P, _P, _P, _P, _i, _i, _i, _i, _i, _i, _P]),
    "lrpx_cam_expand_rows_f32": (_i, [_P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_aoa_decoder_workspace_bytes": (_sz, [C.POINTER(AoaArgs)]),
    "lrpx_aoa_decoder_lrp_f32": (_i, [C.POINTER(AoaArgs), _P, _sz, _P]),
    "lrpx_adaptive_decoder_workspace_bytes": (_sz, [C.POINTER(AdaptiveArgs)]),
    "lrpx_adaptive_decoder_lrp_f32": (_i, [C.POINTER(AdaptiveArgs), _P, _sz, _P]),
    "lrpx_fc_lrp_weights_f32": (_i, [_P, _P, _P, _P, _P, _P, _P, _P, _i, _i, _i, _P]),
    "lrpx_beam_step": (_i, [C.POINTER(BeamArgs), _P]),
    "lrpx_beam_gather_f32": (_i, [C.POINTER(BeamGatherArgs), _P]),
    "lrpx_block_image_f32": (_i, [C.POINTER(BlockImageArgs), _P]),
    "lrpx_bbox_ratio_f32": (_i, [C.POINTER(BboxArgs), _P]),
    "lrpx_lstm_cell_f32": (_i, [C.POINTER(LstmCellArgs), _P]),
    "lrpx_adaptive_attention_f32": (_i, [C.POINTER(AdaAttentionArgs), _P]),
    "lrpx_lstm_prep_weights_f32": (_i, [_P, _P, _i, _i, _i, _P]),
    "lrpx_lstm_step_f32": (_i, [C.POINTER(LstmStepArgs), _P]),
    "lrpx_tc_conv": (_i, [C.POINTER(TcConvArgs), _P]),
    "lrpx_tc_gemm_bf16_f32": (_i, [_P, _P, _P, _i, _i, _i, _P]),
    "lrpx_gemm_x3_workspace_bytes": (_sz, [_i, _i]),
    "lrpx_gemm_x3_f32": (_i, [_P, _i, _P, _i, _P, _P, _i, _i, _i, _i, _P, _sz, _P]),
    "lrpx_weight_prep_bf16": (_i, [_P, _P, _i, _i, _i, _i, _i, _i, _i, _P]),
    "lrpx_tc_first_fwd": (_i, [_P, _P, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_im2col3_split_bf16": (_i, [_P, _P, _i, _i, _i, _P]),
    "lrpx_tc_maxpool2_bf16": (_i, [_P, _P, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_scale_rows": (_i, [_P, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_pf_to_dense_f32": (_i, [_P, _P, _i, _i, _i, _i, _i, _P]),
    "lrpx_tc_nchw_to_pf_bf16": (_i, [_P, _P, _i, _i, _i, _i, _i, _P]),
    "lrpx_tc_im2col3_split_x": (_i, [_P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_maxpool2_x": (_i, [_P, _P, _P, _P, _P, _P, _P, _i, _i, _i, _i, _i, _P]),
    "lrpx_tc_scale_rows_x": (_i, [_P, _P, _P, _P, _P, _i, _i, _i, _i, _i, _i, _P]),
    "lrpx_tc_pf_split_to_dense_f32": (_i, [_P, _P, _i, _i, _i, _i, _i, _P]),
    "lrpx_tc_im2col7s2_split_bf16": (_i, [_P, _P, _i, _i, _i, _P]),
    "lrpx_tc_maxpool3s2_bf16": (_i, [_P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_unpool3s2_bf16": (_i, [_P, _P, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_subsample2_bf16": (_i, [_P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_stem_col2im_f32": (_i, [_P, _i, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_stem_col2im_bf16": (_i, [_P, _i, _P, _P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_im2col7s2_split_x": (_i, [_P, _P, _i, _i, _i, _i, _P]),
    "lrpx_tc_maxpool3s2_x": (_i, [_P, _P, _P, _i, _i, _i, _i, _i, _P]),
}

_lib = None


def lib():
    """Loads liblrpx.so (once).  Raises LrpxError when it has not been built — there is no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LrpxError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (build()) first; "
                            "lrpx has no CPU / PyTorch fallback")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(l, name)          # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


CALLS = {}     # successful C-ABI calls by name (bench.py reports kernel launches from it)


def check(rc, what=""):
    CALLS[what] = CALLS.get(what, 0) + 1
    if rc != 0:
        msg = lib().lrpx_last_error().decode(errors="replace")
        raise LrpxError(f"{what} failed ({rc}): {msg}")
