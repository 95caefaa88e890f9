"""Tensor-core (tcgen05/TMA, bf16) relevance engine for the Bottleneck ResNet encoder (models/resnet.py:95-239).

Same idea as lrpx.tc.TcVggEngine — the forward runs ONCE per image and hoists everything that does not depend on the
explained word into per-image gains, so that an explanation costs one contraction per conv layer — extended to the
rules a residual network adds (LRPtools/lrp_modules.py:197-280, rule selection lrp_wrapper.py:43-56):

  conv (alpha=1, beta=0, no bias)     s = R / safe(z+),  R_in = a (.) (W+^T * s)                   :81-84, utils.py:16-31
  BatchNorm2d (abs-ratio, Q12)        R_in = |x w| / (|x w| + |b|) R_out                            :204-215
  Add (Q14)                           R_i = x_i / (out + 0.01 sign out) R_out  (out == 0: half each) :262-275
  ReLU                                identity                                                       :42-46
  MaxPool2d(3, 2, 1)                  winner-take-all over overlapping windows                      :186-191
  fork at a block input               the relevances of both branches add (autograd does it in the reference)

Per Bottleneck with input x, a1 = relu(bn1(conv1 x)), a2 = relu(bn2(conv2 a1)), y3 = bn3(conv3 a2), idn = x or
bn_d(conv_d x), out = relu(y3 + idn), the per-image gains written by the forward epilogues (LRPX_TC_EPI_FWDX) are
  G1 = a1 ratio1 / z+1,  G2 = a2 ratio2 / z+2,  G3 = rho1 ratio3 / z+3,  Gs = rho2 (x ratio_d / z+_d with a downsample),
  out (.) G3,  out (.) Gs
and the relevance of one request walks, per block, three (four with a downsample) GEMMs whose epilogues
(LRPX_TC_EPI_MULX / MULX_UNPOOL) multiply by those gains:
  A3 = R_out (.) G3  -> conv3^T -> (.) G2 -> conv2^T -> (.) G1 -> conv1^T -> R_x = acc (.) x + [identity-branch relevance]
  and directly  A3' = R_x (.) G3',  S' = R_x (.) Gs'  of the block below (two outputs of ONE epilogue).
Stride-2 convolutions: the forward computes the stride-1 result and keeps the even pixels (epilogue store flag), the
transposed pass zero-stuffs its operand (MULX_UNPOOL with every "winner" at the first pixel of the 2x2 block) and runs the
stride-1 kernel — 4x the minimal MMA work on 3 of the ~100 layers.  The 7x7 / stride-2 stem is a 1x1 GEMM over a
sign-split im2col in the forward and a 1x1 GEMM (K = 64, N = 49 taps x 6) + a gather (col2im) in the relevance pass.
The relevance chain has bf16 operands and storage.  precision='fp32' gives the forward alone with error-compensated
bf16x3 operands (hi|lo activations, fp32 gains), and TcResNetMixed runs that forward under the bf16 chain (precision
'mixed').  The fp32 bar of the chain itself is the CUDA-core rule path of LRPtools (precision 'fp32' / 'simt').
"""
import ctypes as C
from typing import Optional

import torch

from . import _lib
from ._lib import check, lib
from .tc import (EPI_FWDX, EPI_MULX, EPI_MULX_UNPOOL, EPI_STORE_F32, _k_operand, _need_cuda, _ptr, _stream,
                 dual_forward_weights, pf_rows, pf_to_dense, tc_conv, weight_prep)


def _fold_bn(bn):
    w = (bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().float()
    b = (bn.bias - bn.running_mean * bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().float()
    return w.contiguous(), b.contiguous()


def _split_dual_weights(w):
    """dual_forward_weights with error-compensated operands: per tile the W rows and the W+ rows, each laid out
    [hi | hi | lo] along K per tap (the B operand of an A row [hi | lo], a_phys = 2 cin)."""
    cout = w.shape[0]
    half = cout if cout < 128 else 128
    wf = w.detach().float().permute(0, 2, 3, 1)                      # (cout, kh, kw, cin): K ordered (tap, channel)
    ops_ = [_k_operand(t, True).reshape(cout, -1) for t in (wf, wf.clamp(min=0))]
    return torch.cat([o[j * half:(j + 1) * half] for j in range(cout // half) for o in ops_], 0).contiguous()


class _RConv:
    """one conv + its BatchNorm: operands of the forward (rows [W | W+] per tile) and of the transposed pass (W+^T)"""

    def __init__(self, conv, bn, device, split=False):
        w = conv.weight.detach().to(device=device, dtype=torch.float32).contiguous()
        self.cout, self.cin, self.k = int(w.shape[0]), int(w.shape[1]), int(w.shape[2])
        st = conv.stride if isinstance(conv.stride, tuple) else (conv.stride, conv.stride)
        self.stride = int(st[0])
        if conv.bias is not None or conv.groups != 1 or self.k not in (1, 3) or self.cin % 64 or self.cout % 64:
            raise _lib.LrpxError("TcResNetEngine: bias-free 1x1 / 3x3 convolutions with channels in multiples of 64 only")
        self.w_fwd = _split_dual_weights(w) if split else dual_forward_weights(w)     # (2*cout, k*k*cin [x3])
        self.w_rel = weight_prep(w, 2)                            # (cin, k*k*cout): W+ flipped and transposed
        self.bn_w, self.bn_b = (t.to(device) for t in _fold_bn(bn))


class ResNetState:
    def __init__(self):
        self.n = 0
        self.x = None            # fp32 NCHW images
        self.stem = None         # dict: G (ratio / z+ at the stem output), idx (3x3 pool winners), x0 (pool output)
        self.blocks = []         # per block: dict of gains
        self.feat_pf = None
        self.feat_hw = (0, 0)
        self.feat_c = 0


class TcResNetEngine:
    DELIVER = {"full": 0, "channel_mean": 1, "fp16": 2}
    GROUP = 1024                 # requests walked through the blocks at once (bounds the per-request buffers)
    general, rm, km = True, 1, 1

    def __init__(self, model, device=None, precision="bf16"):
        """precision 'bf16': bf16 operands and storage.  'fp32': the forward with error-compensated operands (hi|lo
        activations, a*w ~ a_hi*w_hi + a_lo*w_hi + a_hi*w_lo with K tripled, fp32 gains); this engine's ``relevance``
        then raises (TcResNetMixed runs the bf16 chain on that forward)."""
        device = torch.device(device or "cuda")
        if device.type != "cuda":
            raise _lib.LrpxError("TcResNetEngine needs a CUDA device: lrpx has no CPU fallback")
        if precision not in ("bf16", "fp32"):
            raise _lib.LrpxError("TcResNetEngine: precision must be 'bf16' or 'fp32'")
        self.device = device
        self.precision = precision
        self.split = self.fwd_split = precision == "fp32"
        m = model
        if m.training:
            raise _lib.LrpxError("TcResNetEngine needs eval() mode (running BatchNorm statistics)")
        w = m.conv1.weight.detach().to(device=device, dtype=torch.float32)
        if tuple(w.shape) != (64, 3, 7, 7) or m.conv1.bias is not None:
            raise _lib.LrpxError("TcResNetEngine: the stem must be a bias-free 7x7 convolution 3 -> 64")
        pool = m.maxpool
        pair = lambda v: tuple(v) if isinstance(v, (tuple, list)) else (v, v)
        if pair(pool.kernel_size) != (3, 3) or pair(pool.stride) != (2, 2) or pair(pool.padding) != (1, 1):
            raise _lib.LrpxError("TcResNetEngine: the stem pool must be MaxPool2d(3, 2, 1)")
        w147 = w.reshape(64, 147)
        pad = w147.new_zeros(64, 26)
        self.stem_w_fwd = _k_operand(torch.cat((torch.cat((w147, w147, pad), 1),
                                                torch.cat((w147.clamp(min=0), w147.clamp(max=0), pad), 1)), 0),
                                     self.fwd_split).contiguous()                  # (128, 320), split: (128, 960)
        # transposed pass: row (ky*7+kx)*6 + s*3 + c = W(s)[:, c, ky, kx] over the 64 channels (s = 0: W+, 1: W-), 294 -> 320 rows
        wt = torch.stack((w.clamp(min=0), w.clamp(max=0)), 0)               # (s, ch, c, ky, kx)
        rows = wt.permute(3, 4, 0, 2, 1).reshape(294, 64)
        self.stem_w_rel = torch.cat((rows, rows.new_zeros(26, 64)), 0).to(torch.bfloat16).contiguous()
        self.stem_bn_w, self.stem_bn_b = (t.to(device) for t in _fold_bn(m.bn1))
        self.blocks = []
        for L in (m.layer1, m.layer2, m.layer3, m.layer4):
            for b in L:
                if not all(hasattr(b, a) for a in ("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "add")):
                    raise _lib.LrpxError("TcResNetEngine: Bottleneck blocks with an explicit Add module only")
                sp = self.fwd_split
                blk = dict(c1=_RConv(b.conv1, b.bn1, device, sp), c2=_RConv(b.conv2, b.bn2, device, sp),
                           c3=_RConv(b.conv3, b.bn3, device, sp),
                           down=_RConv(b.downsample[0], b.downsample[1], device, sp) if b.downsample is not None else None)
                blk["stride"] = blk["c2"].stride
                if blk["stride"] not in (1, 2) or blk["c1"].stride != 1 or blk["c3"].stride != 1:
                    raise _lib.LrpxError("TcResNetEngine: stride 1 or 2 on conv2 / the downsample only")
                if blk["down"] is not None and blk["down"].stride != blk["stride"]:
                    raise _lib.LrpxError("TcResNetEngine: the downsample stride must equal conv2's")
                self.blocks.append(blk)
        self.img_hw = None

    # ------------------------------------------------------------------------------------------ forward
    def _fwd(self, a, cv, n, h, w, out, gain, gain_mode=0, **kw):
        if self.fwd_split:
            kw.update(a_phys=2 * cv.cin, split=1)
        tc_conv(a, cv.w_fwd, n, h, w, cv.cin * (3 if self.fwd_split else 1), 2 * cv.cout, cv.k, EPI_FWDX, out, out2=gain,
                bn_w=cv.bn_w, bn_b=cv.bn_b, n_acc=2, gain_mode=gain_mode, **kw)

    def _keep_stem(self, g):
        """what the state keeps of the stem's forward (TcResNetMixed: bf16 copies)"""
        return g

    def _keep_block(self, g):
        """what the state keeps of one block's forward (TcResNetMixed: bf16 copies)"""
        return g

    def forward(self, x: torch.Tensor, keep_act: bool = False) -> ResNetState:
        _need_cuda(x, "x")
        x = x.detach().float().contiguous()
        n, cin, H, W = x.shape
        if cin != 3 or H % 32 or W % 32:
            raise _lib.LrpxError("images must be (n,3,h,w) with h, w divisible by 32")
        dev = x.device
        sp = self.fwd_split
        m = 2 if sp else 1                         # stored bf16 columns per channel of an activation row (hi|lo)
        mk = lambda rows, c, zero, dt: (torch.zeros if zero else torch.empty)(rows, c, device=dev, dtype=dt)
        bf = lambda rows, c, zero=False: mk(rows, m * c, zero, torch.bfloat16)                       # activations
        gn = lambda rows, c, zero=False: mk(rows, c, zero, torch.float32 if sp else torch.bfloat16)  # gains
        st = ResNetState()
        st.n, st.x = n, x
        self.img_hw = (H, W)
        h, w = H // 2, W // 2
        rows = pf_rows(n, h, w)
        cols = bf(rows, 320)
        if sp:
            check(lib().lrpx_tc_im2col7s2_split_x(_ptr(x), _ptr(cols), n, H, W, 1, _stream()), "lrpx_tc_im2col7s2_split_x")
        else:
            check(lib().lrpx_tc_im2col7s2_split_bf16(_ptr(x), _ptr(cols), n, H, W, _stream()), "lrpx_tc_im2col7s2_split_bf16")
        act, G = bf(rows, 64), gn(rows, 64)
        tc_conv(cols, self.stem_w_fwd, n, h, w, 960 if sp else 320, 128, 1, EPI_FWDX, act, out2=G, bn_w=self.stem_bn_w,
                bn_b=self.stem_bn_b, n_acc=2, gain_mode=1, a_phys=640 if sp else 0, split=int(sp))
        del cols
        x0 = bf(pf_rows(n, h // 2, w // 2), 64)
        idx = torch.empty(pf_rows(n, h // 2, w // 2), 64, device=dev, dtype=torch.uint8)
        if sp:
            check(lib().lrpx_tc_maxpool3s2_x(_ptr(act), _ptr(x0), _ptr(idx), n, h, w, 64, 1, _stream()), "lrpx_tc_maxpool3s2_x")
        else:
            check(lib().lrpx_tc_maxpool3s2_bf16(_ptr(act), _ptr(x0), _ptr(idx), n, h, w, 64, _stream()),
                  "lrpx_tc_maxpool3s2_bf16")
        del act
        st.stem = self._keep_stem(dict(G=G, idx=idx, x0=x0, hw=(h, w)))
        del G
        h, w = h // 2, w // 2
        cur = x0
        for blk in self.blocks:
            c1, c2, c3, dn, s = blk["c1"], blk["c2"], blk["c3"], blk["down"], blk["stride"]
            hc, wc = h // s, w // s
            rows, rows_c = pf_rows(n, h, w), pf_rows(n, hc, wc)
            a1, G1 = bf(rows, c1.cout), gn(rows, c1.cout)
            self._fwd(cur, c1, n, h, w, a1, G1)
            a2, G2 = bf(rows_c, c2.cout, s == 2), gn(rows_c, c2.cout, s == 2)
            self._fwd(a1, c2, n, h, w, a2, G2, fwd_flags=2 if s == 2 else 0)
            g = dict(x=cur, G1=G1, G2=G2, hw=(h, w), hwc=(hc, wc))
            if dn is not None:
                xs = cur
                if s == 2:
                    xs = bf(rows_c, dn.cin)           # row-wise copy: hi|lo rows are rows of m * cin channels
                    check(lib().lrpx_tc_subsample2_bf16(_ptr(cur), _ptr(xs), n, h, w, m * dn.cin, _stream()),
                          "lrpx_tc_subsample2_bf16")
                idn, Hd = bf(rows_c, dn.cout), gn(rows_c, dn.cout)
                self._fwd(xs, dn, n, hc, wc, idn, Hd, gain_mode=1, fwd_flags=1)
                g["xs"] = xs
                del xs
            else:
                idn, Hd = cur, None
            out = bf(rows_c, c3.cout)
            G3, Gs, xG3, xGs = (gn(rows_c, c3.cout) for _ in range(4))
            self._fwd(a2, c3, n, hc, wc, out, G3, gain_mode=1, out3=Gs, out4=xG3, out5=xGs, idn=idn, hd=Hd)
            g.update(G3=G3, Gs=Gs, xG3=xG3, xGs=xGs)
            del a1, a2, idn, Hd, G1, G2, G3, Gs, xG3, xGs
            st.blocks.append(self._keep_block(g))
            del g
            cur, h, w = out, hc, wc
        st.feat_pf, st.feat_hw, st.feat_c = cur, (h, w), self.blocks[-1]["c3"].cout
        return st

    def features(self, st: ResNetState, layout="nchw"):
        h, w = st.feat_hw
        if self.fwd_split:
            out = torch.empty((st.n, st.feat_c, h, w) if layout == "nchw" else (st.n, h * w, st.feat_c),
                              device=st.feat_pf.device, dtype=torch.float32)
            check(lib().lrpx_tc_pf_split_to_dense_f32(_ptr(st.feat_pf), _ptr(out), st.n, h, w, st.feat_c,
                                                      1 if layout == "nchw" else 0, _stream()),
                  "lrpx_tc_pf_split_to_dense_f32")
            return out
        return pf_to_dense(st.feat_pf, st.n, h, w, st.feat_c, layout)

    # ------------------------------------------------------------------------------------------ relevance
    def heat_shape(self, Q, deliver="full"):
        H, W = self.img_hw
        if deliver == "channel_mean":
            return (Q, H, W), torch.float32
        return (Q, 3, H, W), (torch.float16 if deliver == "fp16" else torch.float32)

    def _blocks_relevance(self, st, r_feat, rimg, Q, stop_at=0):
        """layers 4..1 for Q requests -> relevance at the stem pool's output (Q, h0, w0, 64) PF bf16
        (``stop_at`` = k > 0: the relevance at the input of block k instead — diagnostics / tests)"""
        dev = r_feat.device
        bf = lambda rows, c: torch.empty(rows, c, device=dev, dtype=torch.bfloat16)
        fh, fw = st.feat_hw
        last = st.blocks[-1]
        C = st.feat_c
        A3, S = bf(pf_rows(Q, fh, fw), C), bf(pf_rows(Q, fh, fw), C)
        for rz, dst in ((last["G3"], A3), (last["Gs"], S)):
            check(lib().lrpx_tc_scale_rows(_ptr(r_feat), _ptr(rz), _ptr(rimg), _ptr(dst), Q, fh, fw, C, _stream()),
                  "lrpx_tc_scale_rows")
        for k in range(len(self.blocks) - 1, -1, -1):
            blk, g = self.blocks[k], st.blocks[k]
            c1, c2, c3, dn, s = blk["c1"], blk["c2"], blk["c3"], blk["down"], blk["stride"]
            (h, w), (hc, wc) = g["hw"], g["hwc"]
            # conv3^T (1x1): (.) G2; a stride-2 conv2 wants its operand zero-stuffed at conv2's input resolution
            A2 = bf(pf_rows(Q, h, w), c2.cout)
            tc_conv(A3, c3.w_rel, Q, hc, wc, c3.cout, c3.cin, 1, EPI_MULX_UNPOOL if s == 2 else EPI_MULX, A2, gain=g["G2"],
                    row_img=rimg)
            # conv2^T (3x3, stride 1 on the stuffed operand): (.) G1
            A1 = bf(pf_rows(Q, h, w), c1.cout)
            tc_conv(A2, c2.w_rel, Q, h, w, c2.cout, c2.cin, 3, EPI_MULX, A1, gain=g["G1"], row_img=rimg)
            del A2
            # identity branch: its relevance at the block input
            if dn is not None:
                add = bf(pf_rows(Q, h, w), dn.cin)
                tc_conv(S, dn.w_rel, Q, hc, wc, dn.cout, dn.cin, 1, EPI_MULX_UNPOOL if s == 2 else EPI_MULX, add,
                        gain=g["xs"], row_img=rimg)
            else:
                add = S
            # conv1^T (1x1): R_x = acc (.) x + add, handed on as the two operands of the block below
            if k > stop_at:
                below = st.blocks[k - 1]
                A3n, Sn = bf(pf_rows(Q, h, w), c1.cin), bf(pf_rows(Q, h, w), c1.cin)
                tc_conv(A1, c1.w_rel, Q, h, w, c1.cout, c1.cin, 1, EPI_MULX, A3n, out2=Sn, gain=below["xG3"],
                        gain2=below["xGs"], gain3=below["G3"], gain4=below["Gs"], add=add, add_pitch=c1.cin, groups=2,
                        row_img=rimg)
                A3, S = A3n, Sn
            else:
                R0 = bf(pf_rows(Q, h, w), c1.cin)
                tc_conv(A1, c1.w_rel, Q, h, w, c1.cout, c1.cin, 1, EPI_MULX, R0, gain=g["x"], add=add, add_pitch=c1.cin,
                        groups=1, row_img=rimg)
                return R0
            del A1, add

    def relevance(self, st: ResNetState, r_feat: torch.Tensor, row_img: Optional[torch.Tensor] = None, chunk: int = 128,
                  out: Optional[torch.Tensor] = None, on_chunk=None, deliver: str = "full") -> torch.Tensor:
        """Image relevance for Q requests.  r_feat: fp32 (Q, h*w, C) pixel-major relevance of the encoder output;
        row_img: int32 (Q,) image of each request (None = identity).  Returns the heat-maps in ``deliver`` format."""
        if self.precision == "fp32":
            raise _lib.LrpxError("TcResNetEngine(precision='fp32') runs the forward only: the relevance chain of a ResNet "
                                 "is bf16 (TcResNetMixed runs it on this forward)")
        _need_cuda(r_feat, "r_feat")
        if deliver not in self.DELIVER:
            raise _lib.LrpxError(f"deliver must be one of {sorted(self.DELIVER)}")
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
        shp, dt = self.heat_shape(Q, deliver)
        if out is None:
            out = torch.empty(shp, device=dev, dtype=dt)
        if tuple(out.shape) != shp or out.dtype != dt:
            raise _lib.LrpxError(f"out must be {shp} {dt} for deliver={deliver!r}")
        H, W = self.img_hw
        h, w = st.stem["hw"]
        chunk = max(1, min(chunk, Q))
        for g0 in range(0, Q, self.GROUP):
            g1 = min(Q, g0 + self.GROUP)
            rimg_g = row_img[g0:g1]
            R0 = self._blocks_relevance(st, r_feat[g0:g1], rimg_g, g1 - g0)
            per = pf_rows(1, h // 2, w // 2) * 64
            for q0 in range(g0, g1, chunk):
                q1 = min(g1, q0 + chunk)
                nq, rimg = q1 - q0, row_img[q0:q1]
                r0 = R0.view(-1)[(q0 - g0) * per:(q1 - g0) * per]
                A = torch.empty(pf_rows(nq, h, w), 64, device=dev, dtype=torch.bfloat16)
                check(lib().lrpx_tc_unpool3s2_bf16(_ptr(r0), _ptr(st.stem["idx"]), _ptr(st.stem["G"]), _ptr(rimg), _ptr(A), nq,
                                                   h, w, 64, _stream()), "lrpx_tc_unpool3s2_bf16")
                # P (one row of 49 taps x 6 per stem output pixel) is an intermediate: bf16 halves its 2 x 2.1 GB per chunk
                P = torch.empty(pf_rows(nq, h, w), 320, device=dev, dtype=torch.bfloat16)
                tc_conv(A, self.stem_w_rel, nq, h, w, 64, 320, 1, EPI_STORE_F32, P, fwd_flags=4)
                check(lib().lrpx_tc_stem_col2im_bf16(_ptr(P), 320, _ptr(st.x), _ptr(rimg), _ptr(out[q0:q1]), nq, H, W,
                                                     self.DELIVER[deliver], _stream()), "lrpx_tc_stem_col2im_bf16")
                del A, P
                if on_chunk is not None:
                    on_chunk(q0, q1)
        return out

    # ------------------------------------------------------------------------------------------ accounting
    def _convs(self):
        H, W = self.img_hw or (224, 224)
        yield (H // 2, W // 2, 3, 64, 7)
        h, w = H // 4, W // 4
        for blk in self.blocks:
            s = blk["stride"]
            yield (h, w, blk["c1"].cin, blk["c1"].cout, 1)
            yield (h // s, w // s, blk["c2"].cin, blk["c2"].cout, 3)
            yield (h // s, w // s, blk["c3"].cin, blk["c3"].cout, 1)
            if blk["down"] is not None:
                yield (h // s, w // s, blk["down"].cin, blk["down"].cout, 1)
            h, w = h // s, w // s

    def flops_per_explanation(self) -> float:
        """Algorithmic FLOPs of one explanation's relevance pass (one contraction per conv layer at its own stride)."""
        return float(sum(2.0 * h * w * ci * co * k * k for h, w, ci, co, k in self._convs()))

    def mma_flops_per_explanation(self) -> float:
        return self.flops_per_explanation()

    def flops_forward_per_image(self) -> float:
        """Forward + z+ (two contractions per layer), K tripled in the error-compensated forward."""
        return 2.0 * self.flops_per_explanation() * (3 if self.fwd_split else 1)


class TcResNetMixed(TcResNetEngine):
    """The per-image FORWARD with error-compensated operands (TcResNetEngine precision 'fp32'), the per-explanation
    chain with bf16 operands and storage (precision 'mixed'), the ResNet twin of lrpx.tc.TcVggMixed.  The encoder
    features the decoder consumes are fp32-accurate, the max-pool winners are the accurate forward's, and the Add-rule
    ratios y3 / (out + 0.01 sign out) are formed from fp32-accurate y3 and identity branch: the gains are rounded to bf16
    ONCE, block by block as the forward produces them (the fp32 gains of a block are dropped before the next block
    runs), instead of being formed from bf16 activations.  The block inputs the chain multiplies by (x, and xs of a
    downsample) are the hi halves of the forward's hi|lo rows."""

    def __init__(self, model, device=None):
        super().__init__(model, device, precision="fp32")
        self.precision, self.split = "mixed", False           # the chain's operands and storage are bf16

    @staticmethod
    def _hi(t):
        return t[:, :t.shape[1] // 2].contiguous()

    def _keep_stem(self, g):
        # x0 (the pool output) reaches the chain as block 0's x: no second copy here
        return dict(g, G=g["G"].to(torch.bfloat16), x0=None)

    def _keep_block(self, g):
        out = dict(g, x=self._hi(g["x"]), **{k: g[k].to(torch.bfloat16) for k in ("G1", "G2", "G3", "Gs", "xG3", "xGs")})
        if "xs" in g:
            out["xs"] = out["x"] if g["xs"] is g["x"] else self._hi(g["xs"])
        return out
