"""torch-tensor front ends of the fp32 C-ABI entry points (include/lrpx.h).

torch is used only for device memory and streams; all arithmetic happens in liblrpx.so.
Every function requires CUDA tensors and raises otherwise (no CPU fallback).
"""
import ctypes as C
import os

import torch

from . import _lib
from ._lib import ConvShape, PoolShape, check, lib


def _pair(v):
    return (v, v) if isinstance(v, int) else tuple(v)


def _f32(t: torch.Tensor, name="tensor") -> torch.Tensor:
    if not t.is_cuda:
        raise _lib.LrpxError(f"{name} must be a CUDA tensor: lrpx has no CPU fallback")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def conv_shape(a, w, stride, padding, dilation) -> ConvShape:
    (sh, sw), (ph, pw), (dh, dw) = _pair(stride), _pair(padding), _pair(dilation)
    n, cin, h, wd = a.shape
    cout, cin_w, kh, kw = w.shape
    if cin_w != cin:
        raise _lib.LrpxError("grouped convolutions are not supported (weight cin != input cin)")
    return ConvShape(n, cin, h, wd, cout, kh, kw, sh, sw, ph, pw, dh, dw)


def conv_out_hw(shp: ConvShape):
    P = (shp.h + 2 * shp.pad_h - shp.dil_h * (shp.kh - 1) - 1) // shp.stride_h + 1
    Q = (shp.w + 2 * shp.pad_w - shp.dil_w * (shp.kw - 1) - 1) // shp.stride_w + 1
    return P, Q


NET_POS, NET_NEG, NET_PLAIN = 0, 1, 2


def conv_forward(a, w, bias=None, stride=1, padding=0, dilation=1, relu=False):
    a, w = _f32(a, "a"), _f32(w, "w")
    bias = _f32(bias) if bias is not None else None
    shp = conv_shape(a, w, stride, padding, dilation)
    P, Q = conv_out_hw(shp)
    out = torch.empty(shp.n, shp.cout, P, Q, device=a.device, dtype=torch.float32)
    check(lib().lrpx_conv_forward_f32(_ptr(a), _ptr(w), _ptr(bias), _ptr(out), C.byref(shp), int(relu), _stream()),
          "lrpx_conv_forward_f32")
    return out


def conv_rule_s(a, w, bias, r_out, stride=1, padding=0, dilation=1, net=NET_POS, want_z=False):
    a, w, r_out = _f32(a, "a"), _f32(w, "w"), _f32(r_out, "r_out")
    bias = _f32(bias) if bias is not None else None
    shp = conv_shape(a, w, stride, padding, dilation)
    P, Q = conv_out_hw(shp)
    if tuple(r_out.shape) != (shp.n, shp.cout, P, Q):
        raise _lib.LrpxError(f"r_out shape {tuple(r_out.shape)} != {(shp.n, shp.cout, P, Q)}")
    s = torch.empty_like(r_out)
    z = torch.empty_like(r_out) if want_z else None
    check(lib().lrpx_conv_rule_s_f32(_ptr(a), _ptr(w), _ptr(bias), _ptr(r_out), _ptr(s), _ptr(z), C.byref(shp), net,
                                     _stream()), "lrpx_conv_rule_s_f32")
    return (s, z) if want_z else s


def conv_rule_rin(a, w, s, stride=1, padding=0, dilation=1, net=NET_POS, scale=1.0, out=None):
    a, w, s = _f32(a, "a"), _f32(w, "w"), _f32(s, "s")
    shp = conv_shape(a, w, stride, padding, dilation)
    acc = out is not None
    if out is None:
        out = torch.empty_like(a)
    check(lib().lrpx_conv_rule_rin_f32(_ptr(a), _ptr(w), _ptr(s), _ptr(out), C.byref(shp), net, float(scale),
                                       int(acc), _stream()), "lrpx_conv_rule_rin_f32")
    return out


def conv_alpha_beta(a, w, bias, r_out, stride=1, padding=0, dilation=1, alpha=1.0, beta=0.0, ignore_bias=True):
    """Conv2d alpha-beta rule (LRPtools/lrp_modules.py:124-152): alpha*R(pos-net) - beta*R(neg-net)."""
    b = None if ignore_bias else bias
    s = conv_rule_s(a, w, b, r_out, stride, padding, dilation, NET_POS)
    r = conv_rule_rin(a, w, s, stride, padding, dilation, NET_POS, alpha)
    if beta != 0.0:
        s = conv_rule_s(a, w, b, r_out, stride, padding, dilation, NET_NEG)
        conv_rule_rin(a, w, s, stride, padding, dilation, NET_NEG, -beta, out=r)
    return r


def conv_epsilon(a, w, bias, r_out, stride=1, padding=0, dilation=1, ignore_bias=True):
    """Conv epsilon rule (Linear rule on the unfolded conv; parity unpinned, see oracle)."""
    b = None if ignore_bias else bias
    s = conv_rule_s(a, w, b, r_out, stride, padding, dilation, NET_PLAIN)
    return conv_rule_rin(a, w, s, stride, padding, dilation, NET_PLAIN, 1.0)


def linear_epsilon(a, w, bias, r_out, ignore_bias=True):
    """Linear epsilon rule (LRPtools/lrp_modules.py:9-24) for a (n,in), w (out,in), r_out (n,out)."""
    a, w, r_out = _f32(a, "a"), _f32(w, "w"), _f32(r_out, "r_out")
    bias = _f32(bias) if (bias is not None and not ignore_bias) else None
    n, fin = a.shape
    fout = w.shape[0]
    r_in = torch.empty_like(a)
    ws = torch.empty(n, fout, device=a.device, dtype=torch.float32)
    check(lib().lrpx_linear_eps_f32(_ptr(a), _ptr(w), _ptr(bias), _ptr(r_out), _ptr(r_in), _ptr(ws), n, fin, fout,
                                    int(ignore_bias), _stream()), "lrpx_linear_eps_f32")
    return r_in


def _pool_shape(x, kernel_size, stride, padding) -> PoolShape:
    (kh, kw) = _pair(kernel_size)
    (sh, sw) = _pair(stride if stride is not None else kernel_size)
    (ph, pw) = _pair(padding)
    n, c, h, w = x.shape
    return PoolShape(n, c, h, w, kh, kw, sh, sw, ph, pw)


def maxpool_forward(x, kernel_size, stride=None, padding=0, return_indices=True):
    x = _f32(x, "x")
    shp = _pool_shape(x, kernel_size, stride, padding)
    oh = (shp.h + 2 * shp.pad_h - shp.kh) // shp.stride_h + 1
    ow = (shp.w + 2 * shp.pad_w - shp.kw) // shp.stride_w + 1
    y = torch.empty(shp.n, shp.c, oh, ow, device=x.device, dtype=torch.float32)
    idx = torch.empty(shp.n, shp.c, oh, ow, device=x.device, dtype=torch.int64) if return_indices else None
    check(lib().lrpx_maxpool_forward_f32(_ptr(x), _ptr(y), _ptr(idx), C.byref(shp), _stream()),
          "lrpx_maxpool_forward_f32")
    return (y, idx) if return_indices else y


def maxpool_wta(x, r_out, kernel_size, stride=None, padding=0):
    x, r_out = _f32(x, "x"), _f32(r_out, "r_out")
    shp = _pool_shape(x, kernel_size, stride, padding)
    r_in = torch.empty_like(x)
    check(lib().lrpx_maxpool_wta_f32(_ptr(x), _ptr(r_out), _ptr(r_in), C.byref(shp), _stream()), "lrpx_maxpool_wta_f32")
    return r_in


def avgpool_prop(x, r_out, kernel_size, stride=None, padding=0):
    x, r_out = _f32(x, "x"), _f32(r_out, "r_out")
    shp = _pool_shape(x, kernel_size, stride, padding)
    r_in = torch.empty_like(x)
    check(lib().lrpx_avgpool_prop_f32(_ptr(x), _ptr(r_out), _ptr(r_in), C.byref(shp), _stream()),
          "lrpx_avgpool_prop_f32")
    return r_in


def bn_absratio(x, r_out, running_mean, running_var, gamma, beta, eps):
    x, r_out = _f32(x, "x"), _f32(r_out, "r_out")
    n, c = x.shape[0], x.shape[1]
    hw = x.numel() // (n * c)
    r_in = torch.empty_like(x)
    check(lib().lrpx_bn_absratio_f32(_ptr(x), _ptr(r_out), _ptr(r_in), _ptr(_f32(running_mean)), _ptr(_f32(running_var)),
                                     _ptr(_f32(gamma)), _ptr(_f32(beta)), float(eps), n, c, hw, _stream()),
          "lrpx_bn_absratio_f32")
    return r_in


def add_split(x1, x2, r_out):
    x1, x2, r_out = _f32(x1, "x1"), _f32(x2, "x2"), _f32(r_out, "r_out")
    r1, r2 = torch.empty_like(x1), torch.empty_like(x2)
    if x1.numel() == 0:
        return r1, r2
    check(lib().lrpx_add_split_f32(_ptr(x1), _ptr(x2), _ptr(r_out), _ptr(r1), _ptr(r2), x1.numel(), _stream()),
          "lrpx_add_split_f32")
    return r1, r2


def relu_mask(x, r_out):
    x, r_out = _f32(x, "x"), _f32(r_out, "r_out")
    r_in = torch.empty_like(r_out)
    if x.numel() == 0:
        return r_in
    check(lib().lrpx_relu_mask_f32(_ptr(x), _ptr(r_out), _ptr(r_in), x.numel(), _stream()), "lrpx_relu_mask_f32")
    return r_in


def normalize_relevance(x, temperature=1.0):
    x = _f32(x, "x")
    cols = x.shape[-1]
    rows = x.numel() // cols
    y = torch.empty_like(x)
    if x.numel() == 0:
        return y
    check(lib().lrpx_normalize_relevance_f32(_ptr(x), _ptr(y), rows, cols, float(temperature), _stream()),
          "lrpx_normalize_relevance_f32")
    return y


def sum_f64(x) -> torch.Tensor:
    x = _f32(x, "x")
    out = torch.zeros(1, device=x.device, dtype=torch.float64)
    if x.numel() == 0:
        return out
    check(lib().lrpx_sum_f64(_ptr(x), x.numel(), _ptr(out), _stream()), "lrpx_sum_f64")
    return out


def fc_lrp_weights(logits, h, ctx, fc_weight, is_stop):
    """Batched get_lrp_weight_step (gridTDmodel.py:549-578).  is_stop: uint8/bool (V,) device mask."""
    logits, h, ctx, fc_weight = _f32(logits, "logits"), _f32(h, "h"), _f32(ctx, "ctx"), _f32(fc_weight, "fc")
    if not is_stop.is_cuda:
        raise _lib.LrpxError("is_stop must be a CUDA tensor")
    stop = is_stop.to(torch.uint8).contiguous()
    B, V = logits.shape
    H = h.shape[1]
    w_ctx, w_h = torch.empty_like(h), torch.empty_like(h)
    am = torch.empty(B, device=h.device, dtype=torch.int32)
    check(lib().lrpx_fc_lrp_weights_f32(_ptr(logits), _ptr(h), _ptr(ctx), _ptr(fc_weight), _ptr(stop), _ptr(w_ctx),
                                        _ptr(w_h), _ptr(am), B, V, H, _stream()), "lrpx_fc_lrp_weights_f32")
    return w_ctx, w_h, am


def _fill_args(struct, fields: dict, keep: list):
    for k, v in fields.items():
        if torch.is_tensor(v):
            keep.append(v)
            setattr(struct, k, v.data_ptr())
        elif v is None:
            setattr(struct, k, None)
        else:
            setattr(struct, k, v)
    return struct


DEC_TC_GEMM = 1


class LinearX3:
    """A Linear layer / GEMM at fp32 accuracy on the tensor cores (``lrpx_gemm_x3_f32``: error-compensated bf16x3
    operands, fp32 accumulation): y = x @ W^T + b for W (n, k) as nn.Linear stores it.  The weight is split once
    ([hi | hi | lo] rows, zero-padded to the tile width) and re-split when the source tensor changes.  Shapes the
    kernel does not take (k % 64, n % 4) are refused at construction — callers keep such layers on ``torch.addmm``."""

    def __init__(self, weight, bias=None):
        self.src = (weight, bias)
        self._split = WeightCache()
        n, k = weight.shape
        if k % 64 or n % 4:
            raise _lib.LrpxError("LinearX3: in_features must be a multiple of 64 and out_features a multiple of 4")
        self.n, self.k = int(n), int(k)
        self.n_pad = (self.n + 31) // 32 * 32 if self.n <= 256 else (self.n + 255) // 256 * 256

    @staticmethod
    def supports(weight):
        return weight.shape[1] % 64 == 0 and weight.shape[0] % 4 == 0

    def _prep(self):
        w, b = self.src

        def split():
            wf = w.detach().float()
            if self.n_pad != self.n:
                wf = torch.cat((wf, wf.new_zeros(self.n_pad - self.n, self.k)), 0)
            hi = wf.to(torch.bfloat16)
            lo = (wf - hi.float()).to(torch.bfloat16)
            return torch.cat((hi, hi, lo), 1).contiguous(), None if b is None else b.detach().float().contiguous()
        return self._split.get([t for t in self.src if t is not None], split)

    def __call__(self, x, out=None):
        """x (m, k) fp32 CUDA (rows may be strided: pitch = x.stride(0)) -> (m, n) fp32"""
        if not x.is_cuda:
            raise _lib.LrpxError("LinearX3 needs CUDA tensors: lrpx has no CPU fallback")
        w3, b = self._prep()
        if x.dtype != torch.float32 or x.stride(-1) != 1 or x.stride(0) % 4 or x.data_ptr() % 16:
            x = x.float().contiguous()
        m = x.shape[0]
        if out is None:
            out = torch.empty(m, self.n, device=x.device, dtype=torch.float32)
        nbytes = lib().lrpx_gemm_x3_workspace_bytes(m, self.k)
        ws = torch.empty(nbytes, device=x.device, dtype=torch.uint8)
        check(lib().lrpx_gemm_x3_f32(_ptr(x), x.stride(0), _ptr(w3), self.n_pad, _ptr(b), _ptr(out), out.stride(0), m, self.n,
                                     self.k, _ptr(ws), nbytes, _stream()), "lrpx_gemm_x3_f32")
        return out


def lrp_linear_eps(r_out, forward_input, forward_output, weight):
    """The explainers' vector epsilon rule (gridTDmodel.py:744-765) on the device: r_out (n_out,) or (1,n_out),
    forward_input (n_in,), forward_output (n_out,) or False (recomputed as W x), weight (n_out,n_in) -> (n_in,)."""
    for t, n in ((r_out, "r_out"), (forward_input, "forward_input"), (weight, "weight")):
        if not t.is_cuda:
            raise _lib.LrpxError(f"lrp_linear_eps: {n} must be a CUDA tensor (lrpx has no CPU fallback)")
    W = _f32(weight, "weight")
    n_out, n_in = W.shape
    r = _f32(r_out.reshape(-1), "r_out")
    x = _f32(forward_input.reshape(-1), "forward_input")
    if r.numel() != n_out or x.numel() != n_in:
        raise _lib.LrpxError("lrp_linear_eps: shapes do not match the weight")
    z = None
    if not isinstance(forward_output, bool):
        z = _f32(forward_output.reshape(-1), "forward_output")
        if z.numel() != n_out:
            raise _lib.LrpxError("lrp_linear_eps: forward_output must have n_out elements")
    out = torch.empty(n_in, device=W.device, dtype=torch.float32)
    nbytes = lib().lrpx_lrp_linear_eps_workspace_bytes(n_out, n_in)
    ws = torch.empty(nbytes, device=W.device, dtype=torch.uint8)
    check(lib().lrpx_lrp_linear_eps_f32(_ptr(r), _ptr(x), _ptr(z), _ptr(W), _ptr(out), n_out, n_in, _ptr(ws), nbytes,
                                        _stream()), "lrpx_lrp_linear_eps_f32")
    return out.view_as(forward_input) if forward_input.numel() == n_in else out


def lrp_mha(alpha, value, r_context, context, num_head, head_idx):
    """ExplainAOAAttention.lrp_mha (aoamodel.py:812-862): alpha (heads,P), value (P,H), r_context / context (1,H) or
    (H,) -> (P,H): the value relevance of head ``head_idx``, zeros for the other heads."""
    for t, n in ((alpha, "alpha"), (value, "value"), (r_context, "r_context"), (context, "context")):
        if not t.is_cuda:
            raise _lib.LrpxError(f"lrp_mha: {n} must be a CUDA tensor (lrpx has no CPU fallback)")
    v = _f32(value, "value")
    P, H = v.shape
    a = _f32(alpha, "alpha")
    rc, c = _f32(r_context.reshape(-1), "r_context"), _f32(context.reshape(-1), "context")
    if tuple(a.shape) != (num_head, P) or rc.numel() != H or c.numel() != H:
        raise _lib.LrpxError("lrp_mha: shapes do not match")
    out = torch.empty_like(v)
    check(lib().lrpx_lrp_mha_f32(_ptr(a), _ptr(v), _ptr(rc), _ptr(c), _ptr(out), P, H, int(num_head), int(head_idx),
                                 _stream()), "lrpx_lrp_mha_f32")
    return out


def _check_requests(B, T, V, req_img, req_t, req_word, req_head=None, num_head=0):
    """The decoder kernels index saved state with the request tuples: reject out-of-range requests here (one small
    reduction + read-back; skipped while a CUDA graph is being captured and with LRPX_VALIDATE=0)."""
    if os.environ.get("LRPX_VALIDATE", "1") == "0":
        return
    n = int(req_img.numel())
    if not (int(req_t.numel()) == n and int(req_word.numel()) == n and (req_head is None or int(req_head.numel()) == n)):
        raise _lib.LrpxError("decoder lrp: req_img / req_t / req_word (/ req_head) must have the same length")
    if n == 0 or (req_img.is_cuda and torch.cuda.is_current_stream_capturing()):
        return
    lim = [(req_img, B, "req_img"), (req_t, T, "req_t"), (req_word, V, "req_word")]
    if req_head is not None:
        lim.append((req_head, num_head, "req_head"))
    dev = req_img.device
    stats = torch.stack([torch.stack((v.to(dev).min(), v.to(dev).max())) for v, _, _ in lim]).tolist()
    for (lo, hi), (_, bound, name) in zip(stats, lim):
        if lo < 0 or hi >= bound:
            raise _lib.LrpxError(f"decoder lrp: {name} out of range [0, {bound}): min {int(lo)}, max {int(hi)}")


DEC_W3_READY = 4          # LRPX_DEC_W3_READY


def weight_stamp(tensors):
    """(data pointer, in-place version counter) of each tensor: changes when a tensor is replaced or updated in place
    (``load_state_dict``, an optimizer step, ``p.add_()``).  Caches of prepared weight copies are keyed on it."""
    return tuple((t.data_ptr(), t._version) for t in tensors)


class WeightCache:
    """One value built from some source tensors (prepared weight copies, an engine holding converted weights).
    ``get(sources, build, extra_key)`` runs ``build()`` under no_grad the first time and whenever ``extra_key +
    weight_stamp(sources)`` changes; while the key holds it returns the same object: callers compare it by ``is``, and
    captured CUDA graphs point into it."""

    def __init__(self):
        self.key = self.value = None

    def get(self, sources, build, extra_key=()):
        key = tuple(extra_key) + weight_stamp(sources)
        if key != self.key:
            with torch.no_grad():
                self.value = build()
            self.key = key
        return self.value


def _decoder_workspace(ws_cache, kind, dims, nbytes, dev, tc_gemm, weights=None):
    """Workspace of one LRP-decoder call -> (ws, extra flags, key to store it under after a successful call).
    ``ws_cache`` (a dict owned by the caller — BatchExplainer keeps one next to its weights) makes the workspace
    persistent per argument shape and weights, so the split bf16 copies of the weight matrices written by the first call
    are reused (LRPX_DEC_W3_READY: four conversion kernels less per call).  With ``weights`` (the decoder entry points
    always pass theirs) the key also holds the weights' ``weight_stamp``: other weight tensors, or the same ones updated
    in place, get a workspace of their own.  Entries are never evicted — a captured CUDA graph may point into them — and
    at most four are kept; nothing allocated during a stream capture is cached."""
    ws = None
    key = (kind, dims, nbytes)
    if weights is not None:
        key += (weight_stamp(weights[k] for k in sorted(weights)),)
    if ws_cache is not None and tc_gemm:
        ws = ws_cache.get(key)
        if ws is not None:
            return ws, DEC_W3_READY, None
    ws = torch.empty(max(nbytes, 4), device=dev, dtype=torch.uint8)
    if ws_cache is None or not tc_gemm or len(ws_cache) >= 4 or torch.cuda.is_current_stream_capturing():
        return ws, 0, None
    return ws, 0, key


def _decoder_call(run, size, args_cls, dims, flags, state, state_keys, weights, weight_keys, reqs, want_raw, out,
                  ws_cache=None, ws_kind=None):
    """Shared body of the six batched decoder entry points.  ``dims``: the dimension fields of ``args_cls`` in the order
    B, T, H, E, P, C, V, Q[, num_head]; ``reqs``: req_img, req_t, req_word[, req_head].  Checks the requests, fills the
    args struct with the float32 ``state_keys`` / ``weight_keys`` tensors, the int32 requests and the outputs (``out``
    (Q,P,C), r_words (Q,T)[, r_words_raw]), sizes the workspace with the lib function ``size``, calls ``run``.
    ``ws_kind`` names the decoder in the ``ws_cache`` key (_decoder_workspace).  Returns out, r_words[, r_words_raw]."""
    dev = state["feat"].device
    Q, T = dims["Q"], dims["T"]
    _check_requests(dims["B"], T, dims["V"], *reqs.values(), num_head=dims.get("num_head", 0))
    f = {k: _f32(state[k], k) for k in state_keys}
    f.update({k: _f32(weights[k], k) for k in weight_keys})
    f.update({k: v.to(device=dev, dtype=torch.int32).contiguous() for k, v in reqs.items()})
    res = torch.empty(Q, dims["P"], dims["C"], device=dev, dtype=torch.float32)
    r_words = torch.zeros(Q, T, device=dev, dtype=torch.float32)
    r_raw = torch.zeros(Q, T, device=dev, dtype=torch.float32) if want_raw else None
    f.update({out: res, "r_words": r_words, "r_words_raw": r_raw})
    keep = []
    a = _fill_args(args_cls(**dims, flags=flags), f, keep)
    nbytes = getattr(lib(), size)(C.byref(a))
    ws, extra, store = _decoder_workspace(ws_cache, ws_kind, tuple(dims.values()), nbytes, dev,
                                          bool(flags & DEC_TC_GEMM), weights)
    a.flags |= extra
    check(getattr(lib(), run)(C.byref(a), _ptr(ws), nbytes, _stream()), run)
    if store is not None:
        ws_cache[store] = ws
    return (res, r_words, r_raw) if want_raw else (res, r_words)


def gridtd_decoder_lrp(state: dict, weights: dict, req_img, req_t, req_word, want_raw=False, tc_gemm=False, ws_cache=None):
    """state: tensors of lrpx_gridtd_args (stacked over B images), weights: W_g1,W_g2,W_fc,W_glob,W_proj.
    tc_gemm: run the GEMMs as error-compensated bf16x3 on the tensor cores (LRPX_DEC_TC_GEMM) instead of fp32
    CUDA cores.  Returns r_feat (Q,P,C), r_words (Q,T)[, r_words_raw]."""
    B, P, Cc = state["feat"].shape
    T, H = state["g1"].shape[1], state["g1"].shape[2]
    E = state["glob_pre"].shape[1]
    V = state["pred"].shape[2]
    Q = int(req_img.numel())
    return _decoder_call(
        "lrpx_gridtd_decoder_lrp_f32", "lrpx_gridtd_decoder_workspace_bytes", _lib.GridTDArgs,
        dict(B=B, T=T, H=H, E=E, P=P, C=Cc, V=V, Q=Q), DEC_TC_GEMM if tc_gemm else 0,
        state, ["feat", "avg", "A_pre", "A", "glob_pre", "x1", "x2", "h1", "c1", "h2", "c2", "g1", "i1", "f1", "g2", "i2",
                "f2", "st", "ctx", "ctx_hat", "alpha", "beta", "pred"],
        weights, ["W_g1", "W_g2", "W_fc", "W_glob", "W_proj"],
        dict(req_img=req_img, req_t=req_t, req_word=req_word), want_raw, "r_feat", ws_cache, "gridtd")


def aoa_decoder_lrp(state: dict, weights: dict, num_head, req_img, req_t, req_word, req_head, want_raw=False,
                    tc_gemm=False, ws_cache=None):
    B, P, Cc = state["feat"].shape
    T, H = state["g"].shape[1], state["g"].shape[2]
    E = state["x"].shape[2] - H
    V = state["pred"].shape[2]
    Q = int(req_img.numel())
    return _decoder_call(
        "lrpx_aoa_decoder_lrp_f32", "lrpx_aoa_decoder_workspace_bytes", _lib.AoaArgs,
        dict(B=B, T=T, H=H, E=E, P=P, C=Cc, V=V, Q=Q, num_head=num_head), DEC_TC_GEMM if tc_gemm else 0,
        state, ["feat", "A_pre", "A", "glob", "value", "x", "h", "c", "g", "i", "ctx", "caoa", "caoa_lin", "alpha",
                "pred"],
        weights, ["W_g", "W_fc", "W_aoa", "W_v", "W_proj"],
        dict(req_img=req_img, req_t=req_t, req_word=req_word, req_head=req_head), want_raw, "r_feat", ws_cache, "aoa")


def adaptive_decoder_lrp(state: dict, weights: dict, req_img, req_t, req_word, want_raw=False, tc_gemm=False, ws_cache=None):
    """ExplainAdaptiveAttention.explain_caption_wordt (adaptiveattention.py:679-771) batched over requests.
    state: tensors of lrpx_adaptive_args (stacked over B images), weights: W_g, W_fc, W_glob, W_proj.
    Returns r_feat (Q,P,C), r_words (Q,T)[, r_words_raw]."""
    B, P, Cc = state["feat"].shape
    T, H = state["g"].shape[1], state["g"].shape[2]
    E = state["z_glob"].shape[1]
    V = state["pred"].shape[2]
    Q = int(req_img.numel())
    return _decoder_call(
        "lrpx_adaptive_decoder_lrp_f32", "lrpx_adaptive_decoder_workspace_bytes", _lib.AdaptiveArgs,
        dict(B=B, T=T, H=H, E=E, P=P, C=Cc, V=V, Q=Q), DEC_TC_GEMM if tc_gemm else 0,
        state, ["feat", "avg", "z_proj", "A", "z_glob", "x", "h", "c", "g", "i", "f", "st", "ctx", "ctx_hat", "alpha",
                "beta", "pred"],
        weights, ["W_g", "W_fc", "W_glob", "W_proj"],
        dict(req_img=req_img, req_t=req_t, req_word=req_word), want_raw, "r_feat", ws_cache, "adaptive")


# ------------------------------------------------------------------------------------------ gradient family (f4)
DEC_GUIDED = 2


def gridtd_decoder_grad(state: dict, weights: dict, req_img, req_t, req_word, guided=False, want_raw=False, tc_gemm=False):
    """ExplainGridTDGradient.explain_caption_wordt (gridTDmodel.py:1424-1508; ``guided``: :1588-1675) batched over
    requests.  state: the explainer forward's tensors incl. the output / sentinel gates (o1, o2, sg); weights: W1 (4H,
    H+2E), W2 (4H, 3H), W_fc, W_glob, W_proj.  Returns d_feat (Q,P,C), r_words (Q,T)[, r_words_raw]."""
    B, P, Cc = state["feat"].shape
    T, H = state["g1"].shape[1], state["g1"].shape[2]
    E = weights["W_glob"].shape[0]
    V = weights["W_fc"].shape[0]
    Q = int(req_img.numel())
    return _decoder_call(
        "lrpx_gridtd_decoder_grad_f32", "lrpx_gridtd_decoder_grad_workspace_bytes", _lib.GridTDGradArgs,
        dict(B=B, T=T, H=H, E=E, P=P, C=Cc, V=V, Q=Q), (DEC_TC_GEMM if tc_gemm else 0) | (DEC_GUIDED if guided else 0),
        state, ["feat", "c1", "c2", "g1", "i1", "f1", "o1", "g2", "i2", "f2", "o2", "sg", "alpha", "beta"],
        weights, ["W1", "W2", "W_fc", "W_glob", "W_proj"],
        dict(req_img=req_img, req_t=req_t, req_word=req_word), want_raw, "d_feat")


def aoa_decoder_grad(state: dict, weights: dict, num_head, req_img, req_t, req_word, req_head, want_raw=False,
                     tc_gemm=False):
    """ExplainAOAGradient.explain_caption_wordt (aoamodel.py:1435-1499) batched over requests.  state: the explainer
    forward's tensors incl. the output gate ``o`` and the gate pre-activation ``caoa_gate``; weights: W_g (4H, E+2H),
    W_fc, W_aoa, W_gate, W_v, W_proj."""
    B, P, Cc = state["feat"].shape
    T, H = state["g"].shape[1], state["g"].shape[2]
    E = weights["W_g"].shape[1] - 2 * H
    V = weights["W_fc"].shape[0]
    Q = int(req_img.numel())
    return _decoder_call(
        "lrpx_aoa_decoder_grad_f32", "lrpx_aoa_decoder_grad_workspace_bytes", _lib.AoaGradArgs,
        dict(B=B, T=T, H=H, E=E, P=P, C=Cc, V=V, Q=Q, num_head=num_head), DEC_TC_GEMM if tc_gemm else 0,
        state, ["c", "g", "i", "f", "o", "caoa_gate", "caoa_lin", "alpha"],
        weights, ["W_g", "W_fc", "W_aoa", "W_gate", "W_v", "W_proj"],
        dict(req_img=req_img, req_t=req_t, req_word=req_word, req_head=req_head), want_raw, "d_feat")


def adaptive_decoder_grad(state: dict, weights: dict, req_img, req_t, req_word, want_raw=False, tc_gemm=False):
    """ExplainAdaptiveGradient.explain_caption_wordt (adaptiveattention.py:965-1021) batched over requests.  state: the
    explainer forward's tensors incl. the output gate ``o`` and the sentinel gate ``sg``; weights: W_g (4H, 2E+H), W_fc,
    W_glob, W_proj."""
    B, P, Cc = state["feat"].shape
    T, H = state["g"].shape[1], state["g"].shape[2]
    E = weights["W_glob"].shape[0]
    V = weights["W_fc"].shape[0]
    Q = int(req_img.numel())
    return _decoder_call(
        "lrpx_adaptive_decoder_grad_f32", "lrpx_adaptive_decoder_grad_workspace_bytes", _lib.AdaptiveGradArgs,
        dict(B=B, T=T, H=H, E=E, P=P, C=Cc, V=V, Q=Q), DEC_TC_GEMM if tc_gemm else 0,
        state, ["c", "g", "i", "f", "o", "sg", "alpha", "beta"],
        weights, ["W_g", "W_fc", "W_glob", "W_proj"],
        dict(req_img=req_img, req_t=req_t, req_word=req_word), want_raw, "d_feat")


def grad_cam(feat, grads, req_img=None, out=None):
    """grad_cam (gridTDmodel.py:1760-1771) for Q requests: feat (B,P,C) encoder output, grads (Q,P,C) its gradient,
    both pixel-major; req_img (Q,) int32 or None (identity).  Returns (Q,P) maps in [0, 1] (in ``out`` when given)."""
    feat, grads = _f32(feat, "feat"), _f32(grads, "grads")
    Q, P, Cc = grads.shape
    if req_img is not None:
        req_img = req_img.to(device=feat.device, dtype=torch.int32).contiguous()
    elif Q != feat.shape[0]:
        raise _lib.LrpxError("grad_cam: req_img is required when requests and images differ in number")
    if out is None:
        out = torch.empty(Q, P, device=feat.device, dtype=torch.float32)
    elif tuple(out.shape) != (Q, P) or out.dtype != torch.float32 or not out.is_contiguous():
        raise _lib.LrpxError(f"grad_cam: out must be a contiguous fp32 ({Q}, {P}) tensor")
    check(lib().lrpx_grad_cam_f32(_ptr(feat), _ptr(grads), _ptr(req_img), _ptr(out), Q, P, Cc, _stream()),
          "lrpx_grad_cam_f32")
    return out


def cam_expand_mul(g, cam, Kh, Kw, out=None):
    """Guided Grad-CAM's product (gridTDmodel.py:1826-1828): g (Q,C,H,W) times the pyramid-expanded cam (Q,h,w);
    Kh (H,h), Kw (W,w) the expansion along each axis (models/_gradient.py::expand_operator)."""
    g, cam, Kh, Kw = _f32(g, "g"), _f32(cam, "cam"), _f32(Kh, "Kh"), _f32(Kw, "Kw")
    Q, Cc, H, W = g.shape
    h, w = cam.shape[1:]
    if tuple(Kh.shape) != (H, h) or tuple(Kw.shape) != (W, w) or cam.shape[0] != Q:
        raise _lib.LrpxError("cam_expand_mul: shapes do not match")
    out = torch.empty_like(g) if out is None else out
    check(lib().lrpx_cam_expand_mul_f32(_ptr(g), _ptr(cam), _ptr(Kh), _ptr(Kw), _ptr(out), Q, Cc, h, w, H, W, _stream()),
          "lrpx_cam_expand_mul_f32")
    return out


def cam_expand_rows(cam, Kh):
    """The y half of cam_expand_mul's expansion: (Q,H,w) = Kh (H,h) @ cam (Q,h,w), in its fmaf order.  With the x half
    (Kw) it is the Guided Grad-CAM factor the tensor-core chain applies in its last epilogue (TcVggEngine.relevance's
    ``cam``)."""
    cam, Kh = _f32(cam, "cam"), _f32(Kh, "Kh")
    Q, h, w = cam.shape
    H = Kh.shape[0]
    if Kh.shape[1] != h:
        raise _lib.LrpxError("cam_expand_rows: shapes do not match")
    out = torch.empty(Q, H, w, device=cam.device, dtype=torch.float32)
    check(lib().lrpx_cam_expand_rows_f32(_ptr(cam), _ptr(Kh), _ptr(out), Q, h, w, H, _stream()), "lrpx_cam_expand_rows_f32")
    return out


# ------------------------------------------------------------------------------------------ explainer forward
def _ld(t):
    """row stride (elements) of a 2-D view whose last dimension is contiguous"""
    if t.stride(-1) != 1:
        raise _lib.LrpxError("last dimension must be contiguous")
    return t.stride(0)


def _gate_outputs(a, g, o, sg):
    """optional extra saved gates (the gradient explainers' state): rows share the stride of g/i/f"""
    for name, t in (("o", o), ("sg", sg)):
        if t is not None:
            if not t.is_cuda or t.dtype != torch.float32 or _ld(t) != _ld(g):
                raise _lib.LrpxError(f"{name} must be an fp32 CUDA view with the row stride of g/i/f")
            setattr(a, name, t.data_ptr())


def lstm_cell(z, c_prev, h, c, g, i, f, gate_pre=None, s=None, h_copy0=None, h_copy1=None, h_copy2=None, s_copy=None,
              o=None, sg=None):
    """lrpx_lstm_cell_f32: all arguments are 2-D fp32 CUDA views (B, H) (z: (B, >=4H)) with contiguous rows; outputs
    are written in place.  h/c share one row stride, g/i/f/s (and the optional o / sg) share one."""
    B, H = c_prev.shape
    for t in (z, c_prev, h, c, g, i, f):
        if not t.is_cuda or t.dtype != torch.float32:
            raise _lib.LrpxError("lstm_cell needs fp32 CUDA tensors: lrpx has no CPU fallback")
    if _ld(h) != _ld(c) or not (_ld(g) == _ld(i) == _ld(f)) or (s is not None and _ld(s) != _ld(g)):
        raise _lib.LrpxError("h/c and g/i/f/s must share their row strides")
    a = _lib.LstmCellArgs(B=B, H=H)
    a.z, a.ldz = z.data_ptr(), _ld(z)
    a.c_prev, a.ld_cprev = c_prev.data_ptr(), _ld(c_prev)
    if gate_pre is not None:
        a.gate_pre, a.ld_gate_pre = gate_pre.data_ptr(), _ld(gate_pre)
        a.s = s.data_ptr()
    a.h, a.c, a.ld_state = h.data_ptr(), c.data_ptr(), _ld(h)
    a.g, a.i, a.f, a.ld_gate = g.data_ptr(), i.data_ptr(), f.data_ptr(), _ld(g)
    for name, ldn, t in (("h_copy0", "ld_copy0", h_copy0), ("h_copy1", "ld_copy1", h_copy1), ("h_copy2", "ld_copy2", h_copy2),
                         ("s_copy", "ld_s_copy", s_copy)):
        if t is not None:
            setattr(a, name, t.data_ptr())
            setattr(a, ldn, _ld(t))
    _gate_outputs(a, g, o, sg)
    check(lib().lrpx_lstm_cell_f32(C.byref(a), _stream()), "lrpx_lstm_cell_f32")


def lstm_prep_weights(w, G):
    """lrpx_lstm_prep_weights_f32: (K, G*H) fp32 row-major -> the [H/4][G][4][K] layout lrpx_lstm_step_f32 reads."""
    w = _f32(w, "w")
    K, GH = w.shape
    out = torch.empty(GH * K, device=w.device, dtype=torch.float32)
    check(lib().lrpx_lstm_prep_weights_f32(_ptr(w), _ptr(out), K, G, GH // G, _stream()), "lrpx_lstm_prep_weights_f32")
    return out


def lstm_step(x, wp, add, G, c_prev, h, c, g, i, f, s=None, h_copy0=None, h_copy1=None, h_copy2=None, s_copy=None,
              o=None, sg=None):
    """lrpx_lstm_step_f32: z = add + x @ W (skinny fp32 GEMM) and the LSTM cell rule in one kernel.  x (B,K) row
    view, wp from lstm_prep_weights, add (B,G*H) rows or a (G*H,) vector; the other arguments as in lstm_cell."""
    B, H = c_prev.shape
    for t in (x, wp, add, c_prev, h, c, g, i, f):
        if not t.is_cuda or t.dtype != torch.float32:
            raise _lib.LrpxError("lstm_step needs fp32 CUDA tensors: lrpx has no CPU fallback")
    if _ld(h) != _ld(c) or not (_ld(g) == _ld(i) == _ld(f)) or (s is not None and _ld(s) != _ld(g)):
        raise _lib.LrpxError("h/c and g/i/f/s must share their row strides")
    a = _lib.LstmStepArgs(B=B, H=H, K=x.shape[1], G=G)
    a.x, a.ldx, a.wp = x.data_ptr(), _ld(x), wp.data_ptr()
    a.add, a.ld_add = add.data_ptr(), (0 if add.dim() == 1 else _ld(add))
    a.c_prev, a.ld_cprev = c_prev.data_ptr(), _ld(c_prev)
    a.h, a.c, a.ld_state = h.data_ptr(), c.data_ptr(), _ld(h)
    a.g, a.i, a.f, a.ld_gate = g.data_ptr(), i.data_ptr(), f.data_ptr(), _ld(g)
    if s is not None:
        a.s = s.data_ptr()
    for name, ldn, t in (("h_copy0", "ld_copy0", h_copy0), ("h_copy1", "ld_copy1", h_copy1), ("h_copy2", "ld_copy2", h_copy2),
                         ("s_copy", "ld_s_copy", s_copy)):
        if t is not None:
            setattr(a, name, t.data_ptr())
            setattr(a, ldn, _ld(t))
    _gate_outputs(a, g, o, sg)
    check(lib().lrpx_lstm_step_f32(C.byref(a), _stream()), "lrpx_lstm_step_f32")


def adaptive_attention(A, img_proj, hs_proj, w_h, s, ctx, ctx_hat, alpha, beta, ctx_hat_copy=None, h=None, W_g=None,
                       W_s=None, b_s=None):
    """lrpx_adaptive_attention_f32 (AdaptiveAttention.forward, gridTDmodel.py:61-103); outputs written in place.
    A (B,P,H), img_proj (B,P,K) contiguous; hs_proj (B,2K) or None (then h (B,H) and the projection weights W_g, W_s
    (K,H), b_s (K) are given and the projections are computed in the kernel); s/ctx/ctx_hat (B,H) row views;
    alpha (B,P); beta (B,)."""
    B, P, H = A.shape
    K = img_proj.shape[2]
    if not (A.is_cuda and A.is_contiguous() and img_proj.is_contiguous() and w_h.is_contiguous()):
        raise _lib.LrpxError("adaptive_attention needs contiguous CUDA tensors")
    if _ld(ctx) != _ld(ctx_hat):
        raise _lib.LrpxError("ctx / ctx_hat must share their row stride")
    a = _lib.AdaAttentionArgs(B=B, P=P, K=K, H=H)
    a.A, a.img_proj, a.w_h = A.data_ptr(), img_proj.data_ptr(), w_h.data_ptr()
    if hs_proj is not None:
        a.hs_proj, a.ld_hs = hs_proj.data_ptr(), _ld(hs_proj)
    else:
        for t in (W_g, W_s, b_s):
            if t is None or not t.is_contiguous() or t.dtype != torch.float32:
                raise _lib.LrpxError("W_g, W_s, b_s must be contiguous fp32 tensors when hs_proj is None")
        a.h, a.ld_h = h.data_ptr(), _ld(h)
        a.W_g, a.W_s, a.b_s = W_g.data_ptr(), W_s.data_ptr(), b_s.data_ptr()
    a.s, a.ld_s = s.data_ptr(), _ld(s)
    a.ctx, a.ctx_hat, a.ld_out = ctx.data_ptr(), ctx_hat.data_ptr(), _ld(ctx)
    a.alpha, a.ld_alpha = alpha.data_ptr(), _ld(alpha)
    a.beta, a.ld_beta = beta.data_ptr(), beta.stride(0)
    if ctx_hat_copy is not None:
        a.ctx_hat_copy, a.ld_copy = ctx_hat_copy.data_ptr(), _ld(ctx_hat_copy)
    check(lib().lrpx_adaptive_attention_f32(C.byref(a), _stream()), "lrpx_adaptive_attention_f32")


# ------------------------------------------------------------------------------------------ device beam search
def beam_step(logits, scores, n_alive, seqs, comp_seqs, comp_len, comp_scores, n_comp, prev_words, src_row, step, end_id):
    """lrpx_beam_step: one step of the reference's beam search bookkeeping (gridTDmodel.py:436-462) for B images x k
    slots, in place on the device state tensors (see include/lrpx.h)."""
    B, k, W = seqs.shape
    for t, dt in ((logits, torch.float32), (scores, torch.float32), (comp_scores, torch.float32), (n_alive, torch.int32),
                  (seqs, torch.int32), (comp_seqs, torch.int32), (comp_len, torch.int32), (n_comp, torch.int32),
                  (prev_words, torch.int64), (src_row, torch.int32)):
        if not t.is_cuda or t.dtype != dt or not t.is_contiguous():
            raise _lib.LrpxError("beam_step needs contiguous CUDA tensors of the documented dtypes: lrpx has no CPU fallback")
    a = _lib.BeamArgs(B=B, k=k, V=logits.shape[1], L=W - 1, step=int(step), end_id=int(end_id))
    for name, t in (("logits", logits), ("scores", scores), ("n_alive", n_alive), ("seqs", seqs), ("comp_seqs", comp_seqs),
                    ("comp_len", comp_len), ("comp_scores", comp_scores), ("n_comp", n_comp), ("prev_words", prev_words),
                    ("src_row", src_row)):
        setattr(a, name, t.data_ptr())
    check(lib().lrpx_beam_step(C.byref(a), _stream()), "lrpx_beam_step")


def beam_gather(src_row, pairs):
    """lrpx_beam_gather_f32: dst[row] = src[src_row[row]] for every (dst, src) pair of 2-D fp32 row views."""
    if len(pairs) > _lib.BEAM_GATHER_MAX:
        raise _lib.LrpxError("too many pairs")
    g = _lib.BeamGatherArgs(n_rows=int(src_row.numel()), n_pairs=len(pairs))
    g.src_row = src_row.data_ptr()
    for e, (dst, src) in enumerate(pairs):
        if not (dst.is_cuda and src.is_cuda and dst.dtype == src.dtype == torch.float32 and dst.shape[1] == src.shape[1]):
            raise _lib.LrpxError("beam_gather needs fp32 CUDA row views of equal width")
        g.dst[e], g.src[e] = dst.data_ptr(), src.data_ptr()
        g.ld_dst[e], g.ld_src[e], g.width[e] = _ld(dst), _ld(src), dst.shape[1]
    check(lib().lrpx_beam_gather_f32(C.byref(g), _stream()), "lrpx_beam_gather_f32")


# ------------------------------------------------------------------------------------------ patch ablation
def block_image(heat, k=20, patch=8, images=None, req_img=None, want_mask=True):
    """lrpx_block_image_f32 (EvaluationExperiments.block_image, evaluation.py:57-80, batched): heat (Q,C,H,W) ->
    mask (Q,H,W) with zeros on the k most relevant patch x patch patches [and masked = mask * images[req_img]]."""
    heat = _f32(heat, "heat")
    Q, Cc, H, W = heat.shape
    a = _lib.BlockImageArgs(Q=Q, C=Cc, H=H, W=W, patch=int(patch), k=int(k))
    a.heat = heat.data_ptr()
    keep = [heat]
    mask = masked = None
    if want_mask:
        mask = torch.empty(Q, H, W, device=heat.device, dtype=torch.float32)
        a.mask = mask.data_ptr()
    if images is not None:
        images = _f32(images, "images")
        a.images, a.img_c = images.data_ptr(), images.shape[1]
        if req_img is not None:
            req_img = req_img.to(device=heat.device, dtype=torch.int32).contiguous()
            a.req_img = req_img.data_ptr()
        masked = torch.empty(Q, images.shape[1], H, W, device=heat.device, dtype=torch.float32)
        a.masked = masked.data_ptr()
    check(lib().lrpx_block_image_f32(C.byref(a), _stream()), "lrpx_block_image_f32")
    return (mask, masked) if images is not None else mask


def bbox_ratio(heat, boxes, n_boxes=None, thresholds=(0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9), negative=False,
               inplace_quirk=True):
    """lrpx_bbox_ratio_f32 (evaluation.py:310-342 as applied by bbox_experiment :398-431): heat (Q,C,H,W), boxes
    (Q,nb,4) int (x0,y0,x1,y1), n_boxes (Q,) or None -> ratio (Q,nb,n_thr): share of the thresholded, max-abs normalised
    positive (``negative``: negative) relevance inside each box.  ``inplace_quirk`` (default, = the reference): the
    reference thresholds its map in place, so after the first box every pair sees the largest threshold used so far."""
    heat = _f32(heat, "heat")
    dev = heat.device
    Q, Cc, H, W = heat.shape
    boxes = boxes.to(device=dev, dtype=torch.int32).contiguous()
    thr = torch.tensor(list(thresholds), dtype=torch.float32, device=dev)
    a = _lib.BboxArgs(Q=Q, C=Cc, H=H, W=W, n_thr=int(thr.numel()), max_boxes=int(boxes.shape[1]),
                      sign=-1.0 if negative else 1.0, inplace_quirk=1 if inplace_quirk else 0)
    ratio = torch.empty(Q, boxes.shape[1], thr.numel(), device=dev, dtype=torch.float32)
    a.heat, a.thresholds, a.boxes, a.ratio = heat.data_ptr(), thr.data_ptr(), boxes.data_ptr(), ratio.data_ptr()
    if n_boxes is not None:
        n_boxes = n_boxes.to(device=dev, dtype=torch.int32).contiguous()
        a.n_boxes = n_boxes.data_ptr()
    check(lib().lrpx_bbox_ratio_f32(C.byref(a), _stream()), "lrpx_bbox_ratio_f32")
    return ratio
