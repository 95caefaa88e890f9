"""Tensor-core (tcgen05/TMA, bf16) encoder relevance engine for VGG-style encoders.

Host side only: torch provides device memory and the stream; every arithmetic step is a liblrpx.so call
(include/lrpx.h, "Tensor-core path").  There is no CPU or PyTorch fallback.

What it replaces in the reference, for an encoder made of conv3x3(pad 1) + ReLU (+ 2x2 max-pool) blocks
(models/vgg.py:62-83, gridTDmodel.py:32-35) under the alpha=1, beta=0 preset (lrp_wrapper.py:7-12):

* ``encoder.compute_lrp(img, target=R)`` (lrp_wrapper.py:63-87) re-runs the forward for every explained word
  and, per conv layer, builds 4 conv clones and runs 4 forward + 4 backward convolutions
  (lrp_modules.py:56-170).  Here the forward runs ONCE per image and also produces, per layer,
  ``gain_l = a_{l+1} / safe(z+_l)``; an explanation then costs one transposed-conv contraction per layer:
  ``s_{l-1} = gain_{l-1} (.) (W+_l^T * s_l)`` with ``s_l = R_{l+1} / safe(z+_l)`` — algebraically the
  reference's ``R_in = a (.) (W+^T (R / z+))`` chain (utils.py:21-31), max-pool winner-take-all
  (lrp_modules.py:186-191) folded into the epilogue through the saved 2-bit argmax.
"""
import ctypes as C
import os
from typing import List, Optional, Sequence

import torch

from . import _lib
from ._lib import TcConvArgs, check, lib

EPI_FWD_GAIN, EPI_MUL, EPI_MUL_UNPOOL, EPI_INPUT, EPI_STORE_F32 = 1, 2, 3, 4, 5
EPI_INPUT3, EPI_MULX, EPI_MULX_UNPOOL, EPI_FWDX = 8, 9, 10, 11


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _need_cuda(t, name):
    if not t.is_cuda:
        raise _lib.LrpxError(f"{name} must be a CUDA tensor: lrpx has no CPU fallback")


def pf_rows(n, h, w):
    return n * (h + 1) * (w + 1)


def tc_conv(a, wt, n_img, h, w, cin, ncol, ksize, epilogue, out, out2=None, bias=None, gain=None, row_img=None,
            pool_idx=None, x=None, gain_mode=0, gain2=None, out3=None, a_phys=0, groups=1, split=0, n_acc=0, rule=0,
            zbias=0, alpha=1.0, beta=0.0, add=None, add_pitch=0, gain3=None, gain4=None, bn_w=None, bn_b=None, idn=None,
            hd=None, out4=None, out5=None, fwd_flags=0, cam_rows=None, cam_kw=None, cam_w=0):
    """Thin wrapper of lrpx_tc_conv (all tensors preallocated by the caller)."""
    args = TcConvArgs(n_img=n_img, h=h, w=w, cin=cin, ncol=ncol, ksize=ksize, epilogue=epilogue, gain_mode=gain_mode,
                      a_phys=a_phys, groups=groups, split=split, n_acc=n_acc, rule=rule, zbias=zbias, alpha=alpha,
                      beta=beta, add_pitch=add_pitch, fwd_flags=fwd_flags, cam_w=cam_w)
    for name, t in (("gain2", gain2), ("out3", out3), ("add", add), ("gain3", gain3), ("gain4", gain4), ("bn_w", bn_w),
                    ("bn_b", bn_b), ("idn", idn), ("hd", hd), ("out4", out4), ("out5", out5), ("cam_rows", cam_rows),
                    ("cam_kw", cam_kw)):
        setattr(args, name, t.data_ptr() if t is not None else None)
    args.a, args.wt = a.data_ptr(), wt.data_ptr()
    args.bias = bias.data_ptr() if bias is not None else None
    args.gain = gain.data_ptr() if gain is not None else None
    args.row_img = row_img.data_ptr() if row_img is not None else None
    args.pool_idx = pool_idx.data_ptr() if pool_idx is not None else None
    args.x = x.data_ptr() if x is not None else None
    args.out = out.data_ptr()
    args.out2 = out2.data_ptr() if out2 is not None else None
    check(lib().lrpx_tc_conv(C.byref(args), _stream()), "lrpx_tc_conv")
    return out


def weight_prep(w, mode, rows_pad=None, chan_pad=None, out=None):
    """lrpx_weight_prep_bf16: fp32 (cout,cin,kh,kw) -> bf16 (rows_pad, kh*kw*chan_pad)."""
    _need_cuda(w, "w")
    w = w.detach().float().contiguous()
    cout, cin, kh, kw = w.shape
    rows, chans = (cin, cout) if mode >= 2 else (cout, cin)
    rows_pad = rows if rows_pad is None else rows_pad
    chan_pad = chans if chan_pad is None else chan_pad
    if out is None:
        out = torch.empty(rows_pad, kh * kw * chan_pad, device=w.device, dtype=torch.bfloat16)
    check(lib().lrpx_weight_prep_bf16(_ptr(w), _ptr(out), cout, cin, kh, kw, mode, rows_pad, chan_pad, _stream()),
          "lrpx_weight_prep_bf16")
    return out


def dual_forward_weights(w):
    """Per tile of ``half`` output channels: the W rows followed by the W+ rows (EPI_FWD_GAIN operand)."""
    cout, cin, kh, kw = w.shape
    half = cout if cout < 128 else 128
    if cout % half:
        raise _lib.LrpxError("output channels must be < 128 or a multiple of 128")
    wt = torch.empty(2 * cout, kh * kw * cin, device=w.device, dtype=torch.bfloat16)
    w = w.detach().float().contiguous()
    for j in range(cout // half):
        sl = w[j * half:(j + 1) * half].contiguous()
        weight_prep(sl, 0, out=wt[2 * j * half:(2 * j + 1) * half])
        weight_prep(sl, 1, out=wt[(2 * j + 1) * half:(2 * j + 2) * half])
    return wt


def nchw_to_pf(x, c_pad=None):
    _need_cuda(x, "x")
    x = x.detach().float().contiguous()
    n, c, h, w = x.shape
    c_pad = c if c_pad is None else c_pad
    out = torch.empty(pf_rows(n, h, w), c_pad, device=x.device, dtype=torch.bfloat16)
    check(lib().lrpx_tc_nchw_to_pf_bf16(_ptr(x), _ptr(out), n, c, h, w, c_pad, _stream()), "lrpx_tc_nchw_to_pf_bf16")
    return out


def pf_to_dense(pf, n, h, w, c, layout="nchw"):
    out = torch.empty((n, c, h, w) if layout == "nchw" else (n, h * w, c), device=pf.device, dtype=torch.float32)
    check(lib().lrpx_tc_pf_to_dense_f32(_ptr(pf), _ptr(out), n, h, w, c, 1 if layout == "nchw" else 0, _stream()),
          "lrpx_tc_pf_to_dense_f32")
    return out


def maxpool2(act, gain, n, h, w, c, want_idx=True):
    dev = act.device
    rows = pf_rows(n, h // 2, w // 2)
    pooled = torch.empty(rows, c, device=dev, dtype=torch.bfloat16)
    idx = torch.empty(rows, c, device=dev, dtype=torch.uint8) if want_idx else None
    gpool = torch.empty(rows, c, device=dev, dtype=torch.bfloat16) if gain is not None else None
    check(lib().lrpx_tc_maxpool2_bf16(_ptr(act), _ptr(gain), _ptr(pooled), _ptr(idx), _ptr(gpool), n, h, w, c,
                                      _stream()), "lrpx_tc_maxpool2_bf16")
    return pooled, idx, gpool


def _hi_lo(t):
    """fp32 -> (hi, lo) bf16 with t ~ hi + lo (16 significant bits)."""
    hi = t.to(torch.bfloat16)
    return hi, (t - hi.float()).to(torch.bfloat16)


def _k_operand(t, split):
    """Weight tensor (..., K) fp32 -> bf16 B operand along K: as is, or [hi | hi | lo] to meet an A row viewed as
    [hi | lo | hi] (lrpx_tc_conv_args.a_phys): a*w ~ a_hi*w_hi + a_lo*w_hi + a_hi*w_lo."""
    if not split:
        return t.to(torch.bfloat16)
    hi, lo = _hi_lo(t)
    return torch.cat((hi, hi, lo), -1)


class _Conv:
    __slots__ = ("cin", "cout", "h", "w", "pool_after", "w_f32", "bias", "w_dual", "w_rel", "w_rel3", "w_fwd", "n_acc",
                 "w_rel_fold")


class VggState:
    """Per-batch forward state shared by all explanations of the batch's images."""

    def __init__(self):
        self.n = 0
        self.x = None           # fp32 NCHW images
        self.gain = []          # per conv: PF bf16 gain at the resolution the relevance chain needs it
        self.gain2 = []         # general modes with two gain groups (beta != 0): the neg-net gains
        self.rz2_last = None
        self.acts = None        # keep_act=True: the PF input activations of every conv (diagnostics)
        self.idx = []           # per conv: uint8 argmax of the pool after it (or None)
        self.rz_last = None     # 1 / safe(z+) of the last conv
        self.feat_pf = None     # encoder output, PF bf16
        self.feat_hw = (0, 0)
        self.feat_c = 0


class TcVggEngine:
    """conv3x3/ReLU/max-pool encoder on the tcgen05 kernels: ``forward`` once per image batch, ``relevance``
    for any number of explanation requests against those images."""

    # rule -> lrpx_tc_conv_args.rule.  'gradient' / 'guided' (SURVEY.md §8 f4) reuse the relevance chain for the plain and
    # the guided-backpropagation input gradient: full weights W^T, gain = the ReLU's derivative [a > 0] (exact in bf16),
    # the max-pool scatter unchanged; 'guided' also clamps the gradient at every ReLU (gridTDmodel.py:1680-1686)
    RULES = {"alpha_beta": 0, "epsilon": 1, "gradient": 2, "guided": 3}

    def __init__(self, weights: Sequence[torch.Tensor], biases: Sequence[Optional[torch.Tensor]], cfg: Sequence,
                 device=None, precision="bf16", alpha=1.0, beta=0.0, ignore_bias=True, rule="alpha_beta"):
        """precision 'bf16': bf16 operands and inter-layer storage.  'fp32': the fp32-accurate mode — operands as
        error-compensated bf16 pairs (x = hi + lo; a*w ~ a_hi*w_hi + a_lo*w_hi + a_hi*w_lo on the same tcgen05 kernels,
        K tripled), fp32 gains, hi|lo inter-layer storage.
        rule 'alpha_beta' (lrp_modules.py:129-150): alpha * R(pos-net) - beta * R(neg-net); beta != 0 doubles K with the
        operand row [alpha*R/z+ | -beta*R/z-] against [W+^T | W-^T].  rule 'epsilon': the Linear rule
        (lrp_modules.py:9-24) on the unfolded conv (the reference's Conv2d raises for it: parity unpinned).
        alpha = 1, beta = 0, bf16, ignore_bias is the specialised fast path (EPI_MUL / EPI_MUL_UNPOOL)."""
        device = torch.device(device or "cuda")
        if device.type != "cuda":
            raise _lib.LrpxError("TcVggEngine needs a CUDA device: lrpx has no CPU fallback")
        if precision not in ("bf16", "fp32") or rule not in self.RULES:
            raise _lib.LrpxError(f"TcVggEngine: precision must be 'bf16' or 'fp32', rule one of {sorted(self.RULES)}")
        if rule == "epsilon" and precision != "fp32":
            # gain = a / (z + 0.01 sign z) with the mixed-sign z = W * a: bf16 operands put an absolute error of
            # ~2^-9 sum|w a| on z, larger than the 0.01 stabiliser wherever z is small — measured rel-L2 0.47 against
            # the oracle.  The z+ gains of the alpha-beta rule are same-sign sums and do not have this problem.
            raise _lib.LrpxError("rule='epsilon' needs precision='fp32' (the epsilon gains are ill-conditioned in bf16)")
        self.device = device
        self.precision, self.rule = precision, rule
        self.rule_id = self.RULES[rule]
        self.alpha, self.beta, self.ignore_bias = float(alpha), float(beta), bool(ignore_bias)
        self.split = precision == "fp32"
        self.groups = 2 if (rule == "alpha_beta" and self.beta != 0.0) else 1
        self.general = not (precision == "bf16" and rule == "alpha_beta" and self.alpha == 1.0 and self.beta == 0.0
                            and self.ignore_bias)
        self.rm = self.groups * (2 if self.split else 1)        # stored channels per logical channel of a chain row
        self.km = self.groups * (3 if self.split else 1)        # GEMM K channels per logical channel
        self.convs: List[_Conv] = []
        k = 0
        for v in cfg:
            if v == "M":
                if not self.convs or self.convs[-1].pool_after:
                    raise _lib.LrpxError("cfg: a pool must follow a conv")
                self.convs[-1].pool_after = True
                continue
            c = _Conv()
            w = weights[k].detach().to(device=device, dtype=torch.float32).contiguous()
            c.cout, c.cin = int(w.shape[0]), int(w.shape[1])
            if tuple(w.shape[2:]) != (3, 3) or c.cout != int(v):
                raise _lib.LrpxError("TcVggEngine supports 3x3 convolutions matching cfg only")
            c.pool_after = False
            c.w_f32 = w
            c.bias = None if biases[k] is None else biases[k].detach().to(device=device, dtype=torch.float32).contiguous()
            c.w_dual = c.w_rel = c.w_rel3 = c.w_fwd = c.w_rel_fold = None
            c.n_acc = 0
            if k == 0 and (c.cin != 3 or c.cout not in (8, 16, 32, 64)):
                raise _lib.LrpxError("first conv must be 3 -> {8,16,32,64} channels")
            if k > 0 and (c.cin % 64 or c.cout % 32):
                raise _lib.LrpxError("conv channels must be multiples of 64 (in) / 32 (out) on the tensor-core path")
            if self.general:
                pass                                     # operands built by _general_weights below
            elif k == 0:
                # rows 0..2: W+ (flipped, transposed), rows 3..5: W-, rows 6..15: zero
                c.w_rel = torch.zeros(16, 9 * c.cout, device=device, dtype=torch.bfloat16)
                weight_prep(w, 2, out=c.w_rel[0:3])
                weight_prep(w, 3, out=c.w_rel[3:6])
                c.w_dual = None
                # LRPX_TC_EPI_INPUT3: filter columns folded into N — row dx*8 + r holds, K-ordered (dy, channel), the
                # weights of tap (dy, dx) of w_rel's row r
                c.w_rel3 = None
                if c.cout % 64 == 0 and os.environ.get("LRPX_TC_INPUT3", "1") != "0":
                    t = c.w_rel[0:8].reshape(8, 3, 3, c.cout)                      # (r, dy, dx, ch)
                    c.w_rel3 = t.permute(2, 0, 1, 3).reshape(24, 3 * c.cout).contiguous()
                if c.cout % 32 == 0:
                    # forward on the tensor cores over the sign-split im2col (lrpx_tc_im2col3_split_bf16):
                    # rows [w | w | 0] -> z, rows [w+ | w- | 0] -> z+   (K = 27 + 27 + 10 zero columns)
                    w27 = w.reshape(c.cout, 27)
                    pad = w27.new_zeros(c.cout, 10)
                    c.w_dual = torch.cat((torch.cat((w27, w27, pad), 1),
                                          torch.cat((w27.clamp(min=0), w27.clamp(max=0), pad), 1)), 0).to(torch.bfloat16).contiguous()
            else:
                c.w_dual = dual_forward_weights(w)
                c.w_rel = weight_prep(w, 2)          # (cin, 9*cout): W+ flipped & transposed
                # 64-column layers without a pool below (VGG16: the 64 -> 64 layer at full resolution) can run with the
                # filter columns folded into N (LRPX_TC_FOLD_COLUMNS: row dx*cin + n, K ordered (filter row, channel)).
                # OFF by default: a third of the MMAs, but the shifted-sum epilogue is one latency-bound pass per
                # 126-row tile and the layer takes 1.25 ms per 128 requests instead of 0.61 (DESIGN.md §7).
                if c.cin == 64 and not self.convs[-1].pool_after and os.environ.get("LRPX_TC_FOLD64", "0") == "1":
                    c.w_rel_fold = (c.w_rel.reshape(c.cin, 3, 3, c.cout).permute(2, 0, 1, 3)
                                    .reshape(3 * c.cin, 3 * c.cout).contiguous())
            if self.general:
                self._general_weights(c, w, first=(k == 0))
            self.convs.append(c)
            k += 1
        if self.convs[-1].pool_after:
            raise _lib.LrpxError("the encoder slice must end with a conv (vgg16.features[0:-1])")

    # ------------------------------------------------------------------------------------------
    def _general_weights(self, c, w, first):
        """B operands of the general modes, laid out on the device once per model (torch tensor ops: not on the
        per-explanation path)."""
        sp, eps = self.split, self.rule != "alpha_beta"       # eps: ONE accumulator of the full weights (also gradient rules)
        grad = self.rule_id >= 2
        pos, neg = (lambda t: t.clamp(min=0)), (lambda t: t.clamp(max=0))
        wt = w.flip(2, 3).permute(1, 2, 3, 0)                    # (cin,3,3,cout): W[co][ci][2-r][2-s]  (transposed conv)
        c.n_acc = 1 if eps else (3 if self.groups == 2 else 2)
        if first:
            if c.cout % 64:
                raise _lib.LrpxError("general modes need a first conv with a multiple of 64 output channels")
            # relevance (EPI_INPUT3): rows 0..2 multiply x+, rows 3..5 multiply x-  (lrp_modules.py:81-84,111-114)
            if grad:
                cp, cn = wt, torch.zeros_like(wt)                # the epilogue returns rows 0..2 as they are
            elif eps:
                cp, cn = wt, wt
            elif self.groups == 2:
                cp, cn = torch.cat((pos(wt), neg(wt)), -1), torch.cat((neg(wt), pos(wt)), -1)
            else:
                cp, cn = pos(wt), neg(wt)
            rows8 = torch.cat((cp, cn, torch.zeros_like(cp[:2])), 0)                   # (8,3,3,G*cout)
            t = _k_operand(rows8, sp)                                                  # (8,3,3,Kl)
            c.w_rel3 = t.permute(2, 0, 1, 3).reshape(24, -1).contiguous()              # row dx*8+r, K = (dy, channel)
            c.w_rel = None
            # forward over the sign-split im2col [x+ taps | x- taps | 0]: z, z+ (pos-net), z- (neg-net)
            w27 = w.reshape(c.cout, 27)
            pad = w27.new_zeros(c.cout, 10)
            blocks = [torch.cat((w27, w27, pad), 1)]
            if not eps:
                blocks.append(torch.cat((pos(w27), neg(w27), pad), 1))
                if self.groups == 2:
                    blocks.append(torch.cat((neg(w27), pos(w27), pad), 1))
        else:
            parts = [wt] if eps else ([pos(wt), neg(wt)] if self.groups == 2 else [pos(wt)])
            c.w_rel = _k_operand(torch.cat(parts, -1), sp).reshape(c.cin, -1).contiguous()    # (cin, 9*Kl)
            c.w_rel3 = None
            wf = w.permute(0, 2, 3, 1)                                                 # (cout,3,3,cin)
            blocks = [wf] if eps else ([wf, pos(wf), neg(wf)] if self.groups == 2 else [wf, pos(wf)])
        cap = {1: 256, 2: 128, 3: 64}[c.n_acc]
        half = min(c.cout, cap)
        if c.cout % half:
            raise _lib.LrpxError(f"output channels must be < {cap} or a multiple of it in this mode")
        ops_ = [_k_operand(b, sp).reshape(c.cout, -1) for b in blocks]
        c.w_fwd = torch.cat([o[j * half:(j + 1) * half] for j in range(c.cout // half) for o in ops_], 0).contiguous()
        c.w_dual = None

    def _forward_general(self, st, x, keep_act):
        n, _, h, w = x.shape
        dev = x.device
        sp, G = self.split, self.groups
        gdt = torch.float32 if sp else torch.bfloat16
        rule = self.rule_id
        act = None
        for li, c in enumerate(self.convs):
            c.h, c.w = h, w
            rows = pf_rows(n, h, w)
            out = torch.empty(rows, c.cout * (2 if sp else 1), device=dev, dtype=torch.bfloat16)
            g0 = torch.empty(rows, c.cout, device=dev, dtype=gdt)
            g1 = torch.empty(rows, c.cout, device=dev, dtype=gdt) if G == 2 else None
            last = li == len(self.convs) - 1
            kw = dict(out2=g0, out3=g1, bias=c.bias, gain_mode=1 if last else 0, split=int(sp), n_acc=c.n_acc, rule=rule,
                      zbias=0 if self.ignore_bias else 1, alpha=self.alpha, beta=self.beta)
            if li == 0:
                cols = torch.empty(rows, 128 if sp else 64, device=dev, dtype=torch.bfloat16)
                check(lib().lrpx_tc_im2col3_split_x(_ptr(x), _ptr(cols), n, h, w, int(sp), _stream()),
                      "lrpx_tc_im2col3_split_x")
                tc_conv(cols, c.w_fwd, n, h, w, 192 if sp else 64, c.n_acc * c.cout, 1, EPI_FWDX, out,
                        a_phys=128 if sp else 0, **kw)
                if keep_act:
                    st.acts.append(None)
            else:
                if keep_act:
                    st.acts.append(act)
                tc_conv(act, c.w_fwd, n, h, w, c.cin * (3 if sp else 1), c.n_acc * c.cout, 3, EPI_FWDX, out,
                        a_phys=2 * c.cin if sp else 0, **kw)
            if c.pool_after:
                prow = pf_rows(n, h // 2, w // 2)
                pooled = torch.empty(prow, out.shape[1], device=dev, dtype=torch.bfloat16)
                idx = torch.empty(prow, c.cout, device=dev, dtype=torch.uint8)
                gp0 = torch.empty(prow, c.cout, device=dev, dtype=gdt)
                gp1 = torch.empty(prow, c.cout, device=dev, dtype=gdt) if G == 2 else None
                check(lib().lrpx_tc_maxpool2_x(_ptr(out), _ptr(g0), _ptr(g1), _ptr(pooled), _ptr(idx), _ptr(gp0),
                                               _ptr(gp1), n, h, w, c.cout, int(sp), _stream()), "lrpx_tc_maxpool2_x")
                act, g0, g1 = pooled, gp0, gp1
                h, w = h // 2, w // 2
                st.idx.append(idx)
            else:
                act = out
                st.idx.append(None)
            st.gain.append(g0)
            st.gain2.append(g1)
        st.rz_last, st.rz2_last = st.gain[-1], st.gain2[-1]
        st.feat_pf, st.feat_hw, st.feat_c = act, (h, w), self.convs[-1].cout
        return st

    def forward(self, x: torch.Tensor, keep_act: bool = False) -> VggState:
        """Activation-producing forward (lrp_wrapper.py:70) + per-layer gains; x is fp32 NCHW (n,3,h,w)."""
        _need_cuda(x, "x")
        x = x.detach().float().contiguous()
        n, cin, h, w = x.shape
        npool = sum(c.pool_after for c in self.convs)
        if cin != 3 or h % (1 << npool) or w % (1 << npool):
            raise _lib.LrpxError("images must be (n,3,h,w) with h, w divisible by 2**(number of pools)")
        st = VggState()
        st.n, st.x = n, x
        if keep_act:
            st.acts = []
        if self.general:
            return self._forward_general(st, x, keep_act)
        dev = x.device
        act = None
        for li, c in enumerate(self.convs):
            c.h, c.w = h, w
            rows = pf_rows(n, h, w)
            out = torch.empty(rows, c.cout, device=dev, dtype=torch.bfloat16)
            gain = torch.empty(rows, c.cout, device=dev, dtype=torch.bfloat16)
            last = li == len(self.convs) - 1
            if li == 0 and c.w_dual is not None:
                cols = torch.empty(rows, 64, device=dev, dtype=torch.bfloat16)
                check(lib().lrpx_tc_im2col3_split_bf16(_ptr(x), _ptr(cols), n, h, w, _stream()),
                      "lrpx_tc_im2col3_split_bf16")
                tc_conv(cols, c.w_dual, n, h, w, 64, 2 * c.cout, 1, EPI_FWD_GAIN, out, out2=gain, bias=c.bias)
            elif li == 0:      # narrow first layer (cout 8 / 16): CUDA cores
                check(lib().lrpx_tc_first_fwd(_ptr(x), _ptr(c.w_f32), _ptr(c.bias), _ptr(out), _ptr(gain), n, h, w,
                                              c.cout, _stream()), "lrpx_tc_first_fwd")
            else:
                tc_conv(act, c.w_dual, n, h, w, c.cin, 2 * c.cout, 3, EPI_FWD_GAIN, out, out2=gain, bias=c.bias,
                        gain_mode=1 if last else 0)
            if keep_act:
                st.acts.append(act if li else None)
            if c.pool_after:
                act, idx, gain = maxpool2(out, gain, n, h, w, c.cout)
                h, w = h // 2, w // 2
                st.idx.append(idx)
            else:
                act = out
                st.idx.append(None)
            st.gain.append(gain)
        st.rz_last = st.gain[-1]
        st.feat_pf, st.feat_hw, st.feat_c = act, (h, w), self.convs[-1].cout
        return st

    def features(self, st: VggState, layout="nchw"):
        """Encoder output as dense fp32: 'nchw' (n,C,h,w) or 'pixel' (n,h*w,C)."""
        h, w = st.feat_hw
        if self.split:
            out = torch.empty((st.n, st.feat_c, h, w) if layout == "nchw" else (st.n, h * w, st.feat_c),
                              device=st.feat_pf.device, dtype=torch.float32)
            check(lib().lrpx_tc_pf_split_to_dense_f32(_ptr(st.feat_pf), _ptr(out), st.n, h, w, st.feat_c,
                                                      1 if layout == "nchw" else 0, _stream()),
                  "lrpx_tc_pf_split_to_dense_f32")
            return out
        return pf_to_dense(st.feat_pf, st.n, h, w, st.feat_c, layout)

    # ------------------------------------------------------------------------------------------
    DELIVER = {"full": 0, "channel_mean": 1, "fp16": 2}

    def heat_shape(self, Q, deliver="full"):
        """(shape, dtype) of the heat-maps of Q requests in delivery format ``deliver``: 'full' = fp32 (Q,3,H,W), the
        reference's return value; 'channel_mean' = fp32 (Q,H,W), what evaluation.py:134,411,503 reduce every heat-map
        to first (torch.mean(relevance, dim=(0,1))); 'fp16' = (Q,3,H,W) half.  Formed in the last layer's epilogue."""
        H, W = self.convs[0].h, self.convs[0].w
        if deliver == "channel_mean":
            return (Q, H, W), torch.float32
        return (Q, 3, H, W), (torch.float16 if deliver == "fp16" else torch.float32)

    def relevance(self, st: VggState, r_feat: torch.Tensor, row_img: Optional[torch.Tensor] = None,
                  chunk: int = 128, out: Optional[torch.Tensor] = None, on_chunk=None, deliver: str = "full",
                  cam=None) -> torch.Tensor:
        """Image relevance for Q requests.  r_feat: fp32 (Q, h*w, C) pixel-major relevance of the encoder
        output (what the decoder kernels emit); row_img: int32 (Q,) image of each request (None = identity).
        Returns fp32 (Q, 3, H, W).  ``on_chunk(q0, q1)`` is called after the launches that produce out[q0:q1]
        have been enqueued (used to overlap the device->host copy of finished heat-maps with the next chunk).
        ``cam=(T, Kw)`` (rule 'guided' only): Guided Grad-CAM — every request's image gradient is multiplied by its
        expanded Grad-CAM map in the last layer's epilogue, T = ops.cam_expand_rows(cam maps, Kh) (Q, H, w) and Kw the
        (W, w) expansion along x; the 'full' result equals ops.cam_expand_mul of the plain one bit for bit.
        = ``relevance_tail(relevance_head(...))`` per group of at most ``GROUP`` requests (the stage-1 buffers of a
        group stay within their memory budget however many requests a call brings)."""
        Q = r_feat.shape[0]
        if deliver not in self.DELIVER:
            raise _lib.LrpxError(f"deliver must be one of {sorted(self.DELIVER)}")
        self._check_cam(cam, Q)
        if Q <= self.GROUP:
            head = self.relevance_head(st, r_feat, row_img, chunk)
            return self.relevance_tail(st, head, out=out, on_chunk=on_chunk, deliver=deliver, cam=cam)
        _need_cuda(r_feat, "r_feat")
        if row_img is None:
            if Q != st.n:
                raise _lib.LrpxError("row_img is required when the number of requests differs from the images")
            row_img = torch.arange(Q, device=r_feat.device, dtype=torch.int32)
        if out is None:
            shp, dt = self.heat_shape(Q, deliver)
            out = torch.empty(shp, device=r_feat.device, dtype=dt)
        group = max(chunk, self.GROUP // max(1, chunk) * chunk)
        for g0 in range(0, Q, group):
            g1 = min(Q, g0 + group)
            head = self.relevance_head(st, r_feat[g0:g1], row_img[g0:g1], chunk)
            cb = None if on_chunk is None else (lambda q0, q1, g0=g0: on_chunk(g0 + q0, g0 + q1))
            self.relevance_tail(st, head, out=out[g0:g1], on_chunk=cb, deliver=deliver,
                                cam=None if cam is None else (cam[0][g0:g1], cam[1]))
        return out

    def _check_cam(self, cam, Q):
        """``cam=(T, Kw)`` of relevance / relevance_tail: the guided rule of the general chain, (Q, H, w) and (W, w) fp32"""
        if cam is None:
            return
        if not self.general or self.rule != "guided":
            raise _lib.LrpxError("cam= (Guided Grad-CAM's factor) needs the 'guided' rule of the general chain")
        T, Kw = cam
        H, W = self.convs[0].h, self.convs[0].w
        w = Kw.shape[-1]
        if (tuple(T.shape) != (Q, H, w) or tuple(Kw.shape) != (W, w) or T.dtype != torch.float32
                or Kw.dtype != torch.float32 or not T.is_contiguous() or not Kw.is_contiguous()):
            raise _lib.LrpxError(f"cam must be ((Q, H, w), (W, w)) contiguous fp32 tensors with Q={Q}, H={H}, W={W}")
        _need_cuda(T, "cam rows")
        _need_cuda(Kw, "cam Kw")

    GROUP = 2048          # requests per stage-1 group

    def _run_layers(self, st, s, nq, rimg, lo, hi, bufs, cur):
        """layers hi-1 .. lo (lo >= 1) on nq requests; returns (tensor holding the result, index of its buffer)"""
        for li in range(hi - 1, lo - 1, -1):
            c, below = self.convs[li], self.convs[li - 1]
            dst = bufs[cur ^ 1]
            if self.general:
                tc_conv(s, c.w_rel, nq, c.h, c.w, c.cout * self.km, c.cin, 3,
                        EPI_MULX_UNPOOL if below.pool_after else EPI_MULX, dst, gain=st.gain[li - 1],
                        gain2=st.gain2[li - 1], row_img=rimg, pool_idx=st.idx[li - 1] if below.pool_after else None,
                        a_phys=c.cout * self.rm if self.split else 0, groups=self.groups, split=int(self.split),
                        rule=self.rule_id)
            elif below.pool_after:
                tc_conv(s, c.w_rel, nq, c.h, c.w, c.cout, c.cin, 3, EPI_MUL_UNPOOL, dst, gain=st.gain[li - 1],
                        row_img=rimg, pool_idx=st.idx[li - 1])
            elif c.w_rel_fold is not None:
                tc_conv(s, c.w_rel_fold, nq, c.h, c.w, c.cout, c.cin, 3, EPI_MUL, dst, gain=st.gain[li - 1], row_img=rimg,
                        fwd_flags=8)
            else:
                tc_conv(s, c.w_rel, nq, c.h, c.w, c.cout, c.cin, 3, EPI_MUL, dst, gain=st.gain[li - 1], row_img=rimg)
            cur ^= 1
            s = dst
        return s, cur

    def _scale_rows(self, st, r, rimg, out, nq):
        """chain entry: the top operand row from the decoder's relevance (s = R / z of the last conv)"""
        fh, fw = st.feat_hw
        if self.general:
            check(lib().lrpx_tc_scale_rows_x(_ptr(r), _ptr(st.rz_last), _ptr(st.rz2_last), _ptr(rimg), _ptr(out), nq, fh,
                                             fw, st.feat_c, self.groups, int(self.split) | (2 if self.rule_id == 3 else 0),
                                             _stream()),
                  "lrpx_tc_scale_rows_x")
        else:
            check(lib().lrpx_tc_scale_rows(_ptr(r), _ptr(st.rz_last), _ptr(rimg), _ptr(out), nq, fh, fw, st.feat_c,
                                           _stream()), "lrpx_tc_scale_rows")

    def relevance_head(self, st: VggState, r_feat: torch.Tensor, row_img: Optional[torch.Tensor] = None,
                       chunk: int = 128) -> dict:
        """Stage 1 of ``relevance``: the low-resolution layers over ALL requests in one launch per layer (their tile
        counts per chunk are only ~3 waves of the persistent grid, so chunked launches lose up to a quarter of the
        machine to wave quantisation).  Returns the hand-over for ``relevance_tail``."""
        _need_cuda(r_feat, "r_feat")
        r_feat = r_feat.detach().float().contiguous()
        Q = r_feat.shape[0]
        fh, fw = st.feat_hw
        if tuple(r_feat.shape[1:]) != (fh * fw, st.feat_c):
            raise _lib.LrpxError(f"r_feat must be (Q,{fh * fw},{st.feat_c}), got {tuple(r_feat.shape)}")
        dev = r_feat.device
        if row_img is None:
            if Q != st.n:
                raise _lib.LrpxError("row_img is required when the number of requests differs from the images")
            row_img = torch.arange(Q, device=dev, dtype=torch.int32)
        row_img = row_img.to(device=dev, dtype=torch.int32).contiguous()
        chunk = max(1, min(chunk, Q))
        L = len(self.convs)
        budget = 2 << 30                      # bytes per stage-1 buffer
        n_wide = 0                            # layers L-1 .. L-n_wide handled in stage 1 (their INPUT and OUTPUT fit)
        if Q > chunk:
            for li in range(L - 1, 0, -1):
                c, below = self.convs[li], self.convs[li - 1]
                oh, ow = (2 * c.h, 2 * c.w) if below.pool_after else (c.h, c.w)
                need = max(pf_rows(Q, c.h, c.w) * c.cout, pf_rows(Q, oh, ow) * c.cin) * 2 * self.rm
                if need > budget:
                    break
                n_wide += 1
        split = L - n_wide                    # stage 1 = layers L-1 .. split, stage 2 = layers split-1 .. 0
        s_all = None
        if n_wide > 0:
            elems = 0
            for li in range(L - 1, split - 1, -1):
                c, below = self.convs[li], self.convs[li - 1]
                oh, ow = (2 * c.h, 2 * c.w) if below.pool_after else (c.h, c.w)
                elems = max(elems, pf_rows(Q, c.h, c.w) * c.cout, pf_rows(Q, oh, ow) * c.cin)
            wide = [torch.empty(elems * self.rm, device=dev, dtype=torch.bfloat16) for _ in range(2)]
            self._scale_rows(st, r_feat, row_img, wide[0], Q)
            s_all, _ = self._run_layers(st, wide[0], Q, row_img, split, L, wide, 0)
        return dict(Q=Q, chunk=chunk, split=split, s_all=s_all, r_feat=r_feat, row_img=row_img)

    def relevance_tail(self, st: VggState, head: dict, out: Optional[torch.Tensor] = None, on_chunk=None,
                       deliver: str = "full", cam=None) -> torch.Tensor:
        """Stage 2 of ``relevance``: the high-resolution layers chunk by chunk, ping-ponging two buffers sized for the
        largest layer of a chunk, so that finished heat-maps can leave for the host while the next chunk runs.
        ``cam``: as in ``relevance``."""
        Q, chunk, split, s_all, r_feat, row_img = (head[k] for k in ("Q", "chunk", "split", "s_all", "r_feat", "row_img"))
        self._check_cam(cam, Q)
        dev = r_feat.device
        fh, fw = st.feat_hw
        shp, dt = self.heat_shape(Q, deliver)
        if out is None:
            out = torch.empty(shp, device=dev, dtype=dt)
        if tuple(out.shape) != shp or out.dtype != dt:
            raise _lib.LrpxError(f"out must be {shp} {dt} for deliver={deliver!r}")
        dmode = self.DELIVER[deliver]
        top = self.convs[split - 1]           # first layer of stage 2: its input is (h, w, cout) of that layer
        max_elems = max(pf_rows(chunk, c.h, c.w) * c.cout for c in self.convs[:split]) * self.rm
        buf = [torch.empty(max_elems, device=dev, dtype=torch.bfloat16) for _ in range(2)]
        bounds = list(range(0, Q, chunk)) + [Q]
        if on_chunk is not None and bounds[-1] - bounds[-2] > 32:
            # results are being delivered chunk by chunk (device->host copy under the next chunk's kernels): the copy
            # of the LAST chunk has nothing to hide under, so finish with a short one
            last = bounds[-1] - bounds[-2]
            bounds.insert(-1, bounds[-1] - max(16, last // 4))
        for q0, q1 in zip(bounds[:-1], bounds[1:]):
            nq = q1 - q0
            rimg = row_img[q0:q1]
            if s_all is not None:
                per = pf_rows(1, top.h, top.w) * top.cout * self.rm
                s, cur = s_all[q0 * per:q1 * per], 1      # reads the stage-1 result in place, writes into buf[0]
            else:
                s, cur = buf[0], 0
                self._scale_rows(st, r_feat[q0:q1], rimg, s, nq)
            s, cur = self._run_layers(st, s, nq, rimg, 1, split, buf, cur)
            c0 = self.convs[0]
            if self.general:
                tc_conv(s, c0.w_rel3, nq, c0.h, c0.w, c0.cout * self.km, 24, 3, EPI_INPUT3, out[q0:q1], row_img=rimg,
                        x=st.x, a_phys=c0.cout * self.rm if self.split else 0, gain_mode=dmode, rule=self.rule_id,
                        cam_rows=None if cam is None else cam[0][q0:q1], cam_kw=None if cam is None else cam[1],
                        cam_w=0 if cam is None else cam[1].shape[1])
            elif c0.w_rel3 is not None:
                tc_conv(s, c0.w_rel3, nq, c0.h, c0.w, c0.cout, 24, 3, EPI_INPUT3, out[q0:q1], row_img=rimg, x=st.x,
                        gain_mode=dmode)
            elif dmode:
                raise _lib.LrpxError("deliver != 'full' needs a first conv with a multiple of 64 output channels")
            else:
                tc_conv(s, c0.w_rel, nq, c0.h, c0.w, c0.cout, 16, 3, EPI_INPUT, out[q0:q1], row_img=rimg, x=st.x)
            if on_chunk is not None:
                on_chunk(q0, q1)
        return out

    def conservation(self, st: VggState, r_feat: torch.Tensor, row_img: Optional[torch.Tensor] = None):
        """Diagnostic (north_star: "relevance conservation reported per layer"): [(name, sum R)] from the encoder output
        down to the image, summed over the given requests.  R at the input of conv l is a_l (.) c_l, formed by the SAME
        contraction kernels with the layer's input activation as the gain; needs ``forward(..., keep_act=True)``."""
        if st.acts is None:
            raise _lib.LrpxError("conservation needs the state of forward(x, keep_act=True)")
        r_feat = r_feat.detach().float().contiguous()
        Q = r_feat.shape[0]
        dev = r_feat.device
        if row_img is None:
            row_img = torch.arange(Q, device=dev, dtype=torch.int32)
        row_img = row_img.to(device=dev, dtype=torch.int32).contiguous()
        L = len(self.convs)
        top = self.convs[-1]
        s = torch.empty(pf_rows(Q, top.h, top.w) * top.cout * self.rm, device=dev, dtype=torch.bfloat16)
        self._scale_rows(st, r_feat, row_img, s, Q)
        trace = [("encoder output", float(r_feat.double().sum()))]
        sp = int(self.split)
        for li in range(L - 1, 0, -1):
            c, below = self.convs[li], self.convs[li - 1]
            # R at the input of conv li: acc (.) a_li through the general epilogue with ONE output group
            a = st.acts[li]
            if self.split:
                g = (a[:, :c.cin].float() + a[:, c.cin:].float()).contiguous()
            else:
                g = a
            R = torch.empty(pf_rows(Q, c.h, c.w), c.cin * (2 if self.split else 1), device=dev, dtype=torch.bfloat16)
            tc_conv(s, c.w_rel, Q, c.h, c.w, c.cout * self.km, c.cin, 3, EPI_MULX, R, gain=g, row_img=row_img,
                    a_phys=c.cout * self.rm if self.split else 0, groups=1, split=sp)
            tot = R.double().sum() if not self.split else (R[:, :c.cin].double().sum() + R[:, c.cin:].double().sum())
            trace.append((f"conv{li} input", float(tot)))
            oh, ow = (2 * c.h, 2 * c.w) if below.pool_after else (c.h, c.w)
            nxt = torch.empty(pf_rows(Q, oh, ow) * c.cin * self.rm, device=dev, dtype=torch.bfloat16)
            s, _ = self._run_layers(st, s, Q, row_img, li, li + 1, [None, nxt], 0)
        head = dict(Q=Q, chunk=Q, split=1, s_all=s, r_feat=r_feat, row_img=row_img)
        heat = self.relevance_tail(st, head)
        trace.append(("image", float(heat.double().sum())))
        return trace

    def flops_per_explanation(self) -> float:
        """Algorithmic FLOPs of one explanation's relevance chain (one contraction per conv layer)."""
        return float(sum(2.0 * c.h * c.w * c.cin * c.cout * 9 for c in self.convs))

    def mma_flops_per_explanation(self) -> float:
        """FLOPs the tensor cores execute per explanation in this mode (K x3 for the error-compensated operands,
        x2 for two gain groups)."""
        return self.flops_per_explanation() * self.km

    def flops_forward_per_image(self) -> float:
        """Forward + z+ (two contractions per layer)."""
        return float(sum(4.0 * c.h * c.w * c.cin * c.cout * 9 for c in self.convs))


class TcVggMixed:
    """The per-image FORWARD in the fp32-accurate mode, the per-explanation chain with bf16 operands and storage
    (precision 'mixed'; for the gradient rules this is what precision 'bf16' means).

    * alpha-beta rule (alpha = 1, beta = 0): the encoder features the decoder consumes are fp32-accurate (1e-5 instead of
      the bf16 forward's 7e-3, which the 19-step LSTM chain of the decoder amplifies to a worst request of 9e-2), the
      max-pool winners are the accurate forward's, and the gains a / z+ are rounded to bf16 ONCE instead of being formed
      from bf16 activations; the chain is the specialised bf16 one (EPI_MUL / EPI_MUL_UNPOOL).
    * gradient / guided rules: a gradient is discontinuous in the forward pass — a ReLU whose pre-activation lies within
      the forward's rounding error of zero flips its mask — so a bf16 forward costs the plain gradient far more than the
      bf16 chain does (measured rel-L2 0.33 against autograd with a bf16 forward, 1.8e-2 with this class, the same as the
      fp32-accurate chain).  The masks are 0 / 1 and convert to bf16 exactly.
    The forward runs once per image, the chain once per explanation."""

    def __init__(self, weights, biases, cfg, device=None, rule="alpha_beta"):
        if rule not in ("alpha_beta", "gradient", "guided"):
            raise _lib.LrpxError("TcVggMixed serves the alpha-beta (alpha 1, beta 0), 'gradient' and 'guided' rules")
        self.fwd = TcVggEngine(weights, biases, cfg, device, precision="fp32", rule=rule)
        self.chain = TcVggEngine(weights, biases, cfg, device, precision="bf16", rule=rule)
        self.precision, self.rule = "mixed", rule

    def forward(self, x, keep_act=False):
        src = self.fwd.forward(x, keep_act)
        for cf, cc in zip(self.fwd.convs, self.chain.convs):
            cc.h, cc.w = cf.h, cf.w
        st = VggState()
        st.n, st.x, st.idx = src.n, src.x, src.idx
        st.gain = [g.to(torch.bfloat16) for g in src.gain]          # gradient rules: 0 / 1, exact
        st.gain2 = [None] * len(st.gain)
        st.rz_last, st.rz2_last = st.gain[-1], None
        st.feat_pf, st.feat_hw, st.feat_c = src.feat_pf, src.feat_hw, src.feat_c
        if src.acts is not None:          # keep_act (conservation report): the bf16 head of every hi|lo activation row
            st.acts = [None if a is None else a[:, :a.shape[1] // 2].contiguous() for a in src.acts]
        st.src = src
        return st

    def features(self, st, layout="nchw"):
        return self.fwd.features(st.src, layout)

    def __getattr__(self, name):          # relevance, relevance_head / _tail, heat_shape, convs, flop counters: the chain's
        return getattr(self.chain, name)
