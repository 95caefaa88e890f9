"""Mirror of LRPtools/lrp_wrapper.py (reference :7-87).

The reference abuses the autograd engine as its reverse-topological scheduler: ``add_lrp`` hangs a forward
hook (saves ``module.input``) and a *backward* hook on every leaf, and ``compute_lrp`` calls
``logits.backward(target)`` so that "gradients" between modules are relevances (reference :14-25, :53-55,
:70-80).  Here ``add_lrp`` records an explicit layer plan once and ``compute_lrp`` walks it: a forward that
saves each rule's inputs on the module (same ``module.input`` attribute), then the rule objects of
``lrp_modules`` in reverse — no autograd graph, no discarded true backward (wgrad), no per-call conv clones.
Supported topologies: a Sequential of leaves (the VGG encoder slice) and the Bottleneck ResNet of
models/resnet.py.  Anything else raises ``NotImplementedError`` in ``add_lrp``.
"""
import os
from collections import defaultdict

import torch
import torch.nn as nn

from lrpx import ops
from . import lrp_modules


class SequentialPresetA(object):
    """reference :7-12"""

    def __init__(self):
        self.lrp_params = {"alpha": 1., "beta": 0., "ignore_bias": True}


def get_lrp_hook(lrp_method, lrp_params=None):
    """reference :14-21 — kept for API compatibility (the explicit walker calls the same rule objects)."""
    def lrp_hook(module, relevance_input, relevance_output):
        lrp_module = lrp_modules.get_lrp_module(module)
        return lrp_module.propagate_relevance(module, relevance_input, relevance_output, lrp_method,
                                              lrp_params=lrp_params)
    return lrp_hook


def save_input_hook(module, input_, output):
    """reference :24-25"""
    module.input = input_


class LRPLoss(nn.Module):
    """reference :28-34 — dummy anchor"""

    def forward(self, x):
        return x

    def backward(self, x):
        return x


# ------------------------------------------------------------------------------------------------
def _method_for(module):
    """Rule selection of add_lrp (reference :43-56)."""
    if type(module) in (nn.Linear, nn.BatchNorm2d, nn.BatchNorm1d):
        return 'epsilon'
    if type(module) == nn.ReLU:
        return 'identity'
    return 'alpha_beta'


def _leaf_forward(m, *xs):
    """Forward of one leaf on the CUDA kernels, saving the rule's inputs like save_input_hook."""
    m.input = tuple(xs)
    x = xs[0]
    if isinstance(m, nn.Conv2d):
        if m.groups != 1:
            raise NotImplementedError("grouped convolutions are not supported")
        return ops.conv_forward(x, m.weight.detach(), None if m.bias is None else m.bias.detach(), m.stride,
                                m.padding, m.dilation)
    if isinstance(m, nn.ReLU):
        # an in-place ReLU aliases its saved input in the reference; the identity rule never reads it
        return torch.relu(x)
    if isinstance(m, nn.MaxPool2d):
        return ops.maxpool_forward(x, m.kernel_size, m.stride, m.padding, return_indices=False)
    if isinstance(m, (nn.BatchNorm2d, nn.BatchNorm1d)):
        if m.training:
            raise NotImplementedError("LRP through BatchNorm needs eval() mode (running statistics)")
        shape = [1, -1] + [1] * (x.dim() - 2)
        w = (m.weight / torch.sqrt(m.running_var + m.eps)).detach().view(shape)
        b = (m.bias - m.running_mean * m.weight / torch.sqrt(m.running_var + m.eps)).detach().view(shape)
        return x * w + b
    if isinstance(m, (nn.Dropout, nn.Dropout2d)):
        if m.training:
            raise NotImplementedError("LRP through Dropout needs eval() mode")
        return x
    if isinstance(m, nn.AvgPool2d):
        return torch.nn.functional.avg_pool2d(x, m.kernel_size, m.stride, m.padding)
    if isinstance(m, nn.Linear):
        return torch.nn.functional.linear(x, m.weight.detach(), None if m.bias is None else m.bias.detach())
    if isinstance(m, lrp_modules.resFlatten):
        return x.reshape(x.size(0), -1)
    if isinstance(m, lrp_modules.resAdd):
        return xs[0] + xs[1]
    if isinstance(m, nn.Identity):
        return x
    raise ValueError("Layer type {} not known.".format(type(m)))


def _leaf_backward(m, R):
    if isinstance(m, nn.Identity):
        return (R,)
    rule = lrp_modules.get_lrp_module(m)
    return rule.propagate_relevance(m, None, (R,), m.lrp_method, lrp_params=m.lrp_params)


def _flatten_sequential(model):
    out = []
    for child in model.children():
        if isinstance(child, nn.Sequential):
            out += _flatten_sequential(child)
        elif len(list(child.children())) == 0:
            out.append(child)
        else:
            raise NotImplementedError(f"add_lrp: unsupported container {type(child)} inside a Sequential")
    return out


class _SequentialPlan:
    def __init__(self, model):
        self.leaves = _flatten_sequential(model)

    def forward(self, x):
        for m in self.leaves:
            x = _leaf_forward(m, x)
        return x

    def backward(self, R, trace=None):
        for m in reversed(self.leaves):
            R = _leaf_backward(m, R)[0]
            if trace is not None:
                trace.append((type(m).__name__, float(ops.sum_f64(R).item())))
        return R


class _ResNetPlan:
    """Bottleneck ResNet (models/resnet.py): relevance at the block-input fork is the sum of both branches
    (autograd accumulates it for free in the reference, SURVEY.md Appendix B.4)."""

    def __init__(self, model):
        self.m = model
        self.blocks = [b for L in (model.layer1, model.layer2, model.layer3, model.layer4) for b in L]
        for b in self.blocks:
            if not all(hasattr(b, a) for a in ("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "add")):
                raise NotImplementedError("add_lrp: only Bottleneck blocks with an explicit Add module are supported")

    def forward(self, x):
        m = self.m
        x = _leaf_forward(m.maxpool, _leaf_forward(m.relu, _leaf_forward(m.bn1, _leaf_forward(m.conv1, x))))
        for b in self.blocks:
            o = _leaf_forward(b.relu, _leaf_forward(b.bn1, _leaf_forward(b.conv1, x)))
            o = _leaf_forward(b.relu, _leaf_forward(b.bn2, _leaf_forward(b.conv2, o)))
            o = _leaf_forward(b.bn3, _leaf_forward(b.conv3, o))
            idn = x
            if b.downsample is not None:
                idn = _leaf_forward(b.downsample[1], _leaf_forward(b.downsample[0], x))
            x = _leaf_forward(b.relu, _leaf_forward(b.add, o, idn))
        return x

    def backward(self, R, trace=None):
        m = self.m
        for b in reversed(self.blocks):
            r_o, r_idn = _leaf_backward(b.add, R)          # ReLU after the add: identity rule
            r = _leaf_backward(b.bn3, r_o)[0]
            r = _leaf_backward(b.conv3, r)[0]
            r = _leaf_backward(b.bn2, r)[0]
            r = _leaf_backward(b.conv2, r)[0]
            r = _leaf_backward(b.bn1, r)[0]
            r = _leaf_backward(b.conv1, r)[0]
            if b.downsample is not None:
                rd = _leaf_backward(b.downsample[1], r_idn)[0]
                rd = _leaf_backward(b.downsample[0], rd)[0]
            else:
                rd = r_idn
            R = r + rd
            if trace is not None:
                trace.append(("Bottleneck", float(ops.sum_f64(R).item())))
        R = _leaf_backward(m.maxpool, R)[0]
        R = _leaf_backward(m.bn1, R)[0]
        R = _leaf_backward(m.conv1, R)[0]
        return R


def _tc_cfg(model):
    """The VGG-style layer list the tensor-core engine (lrpx.tc.TcVggEngine) runs: conv3x3/s1/p1 -> ReLU
    [-> max-pool 2x2/s2] blocks ending with a ReLU (models/vgg.py:62-83, gridTDmodel.py:32-35).  -> (convs, cfg) or
    None when the Sequential is anything else (those models stay on the fp32 rule kernels)."""
    if not isinstance(model, nn.Sequential):
        return None
    leaves = _flatten_sequential(model)
    convs, cfg, i = [], [], 0
    pair = lambda v: tuple(v) if isinstance(v, (tuple, list)) else (v, v)
    while i < len(leaves):
        m = leaves[i]
        if not (isinstance(m, nn.Conv2d) and pair(m.kernel_size) == (3, 3) and pair(m.stride) == (1, 1)
                and pair(m.padding) == (1, 1) and pair(m.dilation) == (1, 1) and m.groups == 1
                and m.padding_mode == 'zeros'):
            return None
        if i + 1 >= len(leaves) or type(leaves[i + 1]) != nn.ReLU:
            return None
        convs.append(m)
        cfg.append(m.out_channels)
        i += 2
        if i < len(leaves) and isinstance(leaves[i], nn.MaxPool2d):
            p = leaves[i]
            if not (pair(p.kernel_size) == (2, 2) and pair(p.stride if p.stride is not None else p.kernel_size) == (2, 2)
                    and pair(p.padding) == (0, 0) and pair(p.dilation) == (1, 1) and not p.ceil_mode):
                return None
            cfg.append("M")
            i += 1
    if not convs or cfg[-1] == "M" or convs[0].in_channels != 3 or convs[0].out_channels not in (8, 16, 32, 64):
        return None
    if any(c.in_channels % 64 or c.out_channels % 32 for c in convs[1:]):
        return None
    return convs, cfg


def _is_bottleneck_resnet(model):
    """models/resnet.py ResNet made of Bottleneck blocks with the explicit Add module (what lrpx.tc_resnet runs)."""
    if not all(hasattr(model, a) for a in ("conv1", "bn1", "maxpool", "layer1", "layer2", "layer3", "layer4")):
        return False
    blocks = [b for L in (model.layer1, model.layer2, model.layer3, model.layer4) for b in L]
    return bool(blocks) and all(all(hasattr(b, a) for a in ("conv1", "bn1", "conv2", "bn2", "conv3", "bn3", "add"))
                                for b in blocks)


class _TcResNetPlan:
    """Tensor-core route of ``compute_lrp(precision='bf16' | 'mixed')`` for Bottleneck ResNets (alpha=1, beta=0 preset):
    ONE engine per precision, rebuilt when a parameter or buffer changes (data pointer / in-place version)."""

    def __init__(self, model):
        self.model = model
        self.convs = [m for m in model.modules() if isinstance(m, nn.Conv2d)]
        self._eng = defaultdict(ops.WeightCache)

    def engine(self, precision, lrp_params):
        from lrpx import tc_resnet
        if precision not in ("bf16", "mixed") or float(lrp_params.get("alpha", 1.)) != 1. \
                or float(lrp_params.get("beta", 0.)) != 0. or not lrp_params.get("ignore_bias", True):
            return None
        ps = [p for p in self.model.parameters()] + [b for b in self.model.buffers()]
        cls = tc_resnet.TcResNetMixed if precision == "mixed" else tc_resnet.TcResNetEngine
        return self._eng[precision].get(ps, lambda: cls(self.model, ps[0].device))


class _TcPlan:
    """Tensor-core route of ``compute_lrp`` for VGG-style encoders: ONE TcVggEngine per (precision, alpha, beta),
    rebuilt when a weight tensor changes (data pointer / in-place version)."""

    def __init__(self, convs, cfg):
        self.convs, self.cfg = convs, cfg
        self._eng = defaultdict(ops.WeightCache)

    def engine(self, precision, lrp_params):
        from lrpx import tc
        alpha, beta = float(lrp_params.get("alpha", 1.)), float(lrp_params.get("beta", 0.))
        ignore_bias = bool(lrp_params.get("ignore_bias", True))
        ws = [c.weight for c in self.convs]
        bs = [c.bias for c in self.convs]

        def build():
            if precision == "mixed":          # fp32-accurate forward, bf16 chain (alpha 1 / beta 0 preset only)
                return tc.TcVggMixed(ws, bs, self.cfg, ws[0].device)
            return tc.TcVggEngine(ws, bs, self.cfg, ws[0].device, precision=precision, alpha=alpha, beta=beta,
                                  ignore_bias=ignore_bias)
        return self._eng[precision, alpha, beta, ignore_bias].get(ws + [b for b in bs if b is not None], build)


def _build_plan(model):
    if isinstance(model, nn.Sequential):
        return _SequentialPlan(model)
    if all(hasattr(model, a) for a in ("conv1", "bn1", "maxpool", "layer1", "layer2", "layer3", "layer4")):
        return _ResNetPlan(model)
    raise NotImplementedError(f"add_lrp: unsupported model topology {type(model)}; supported: nn.Sequential of "
                              "leaf layers (VGG encoder) and the Bottleneck ResNet of models/resnet.py")


def add_lrp(model):
    """reference :37-59.  Idempotent (the reference stacks another pair of hooks per call, Q2)."""
    preset = SequentialPresetA()
    for module in model.modules():
        if len(list(module.children())) == 0:
            module.lrp_method = _method_for(module)
            module.lrp_params = preset.lrp_params
    model._lrpx_plan = _build_plan(model)
    tcp = _tc_cfg(model)
    model._lrpx_tc = _TcPlan(*tcp) if tcp is not None else (_TcResNetPlan(model) if _is_bottleneck_resnet(model) else None)
    model.compute_lrp = lambda sample, **kwargs: compute_lrp(model, sample, **kwargs)


# Arithmetic of ``compute_lrp`` when the caller does not say (a keyword the reference does not have):
#   'fp32' — the reference's fp32 bar (rtol 1e-4 / atol 1e-6, scale-relative).  VGG-style encoders run the tcgen05
#            chain with error-compensated bf16x3 operands and fp32 gains / inter-layer storage; every other
#            topology runs the fp32 CUDA-core rule kernels.
#   'bf16' — the tcgen05 chain with bf16 operands and storage (Spearman >= 0.99 / rel-L2 <= 5e-2 vs the reference).
#   'mixed' — fp32-accurate forward (activations, max-pool winners, gains), bf16 chain: lrpx.tc.TcVggMixed, and for
#            Bottleneck ResNets lrpx.tc_resnet.TcResNetMixed (alpha 1 / beta 0 / ignore_bias preset only).
#   'simt' — the fp32 CUDA-core rule kernels whatever the topology (the rule-by-rule walker).
DEFAULT_PRECISION = os.environ.get("LRPX_PRECISION", "fp32")


def compute_lrp(model, sample, target=None, return_output=False, rectify_logits=False, explain_diff=False,
                conservation_trace=None, precision=None):
    """reference :63-87.  ``rectify_logits`` / ``explain_diff`` are accepted and ignored, as there.
    ``precision``: see DEFAULT_PRECISION above.

    Like the reference, the result is accumulated into ``sample.grad`` (the reference never zeroes it, so a
    second call on the same tensor returns the running sum — Q1).  Set LRPX_NO_GRAD_ACCUMULATION=1 to get the
    per-call relevance instead.  ``conservation_trace`` (a list) receives (layer, sum R) pairs.
    """
    if not hasattr(model, "_lrpx_plan"):
        raise RuntimeError("call add_lrp(model) first")
    if not sample.is_cuda:
        raise RuntimeError("lrpx: compute_lrp needs a CUDA tensor (there is no CPU fallback)")
    if target is None:
        raise RuntimeError("grad can be implicitly created only for scalar outputs")   # what .backward(None) raises
    precision = precision or DEFAULT_PRECISION
    if precision not in ("fp32", "bf16", "simt", "mixed"):
        raise ValueError(f"compute_lrp: unknown precision {precision!r}")
    tcp = getattr(model, "_lrpx_tc", None)
    use_tc = tcp is not None and precision in ("fp32", "bf16", "mixed") and conservation_trace is None and sample.dim() == 4
    if use_tc:
        params = tcp.convs[0].lrp_params
        use_tc = all(c.lrp_method == "alpha_beta" and c.lrp_params == params for c in tcp.convs)
        general = not (precision == "bf16" and params.get("alpha", 1.) == 1. and params.get("beta", 0.) == 0.
                       and params.get("ignore_bias", True))
        preset = params.get("alpha", 1.) == 1. and params.get("beta", 0.) == 0. and params.get("ignore_bias", True)
        if precision == "mixed":
            use_tc = use_tc and preset and (isinstance(tcp, _TcResNetPlan) or tcp.convs[0].out_channels % 64 == 0)
        if isinstance(tcp, _TcResNetPlan):
            # ResNets: the bf16 chain only, on the bf16 ('bf16') or the fp32-accurate ('mixed') forward
            use_tc = use_tc and (not general or precision == "mixed") and not model.training
        elif general and tcp.convs[0].out_channels % 64:
            use_tc = False                    # the general kernels need a 64-channel first layer: CUDA-core walker
    if precision in ("bf16", "mixed") and not use_tc:
        raise NotImplementedError(f"compute_lrp(precision={precision!r}): the tensor-core chain covers VGG-style encoders "
                                  "(conv3x3/ReLU/max-pool 2x2) under the alpha-beta rule and Bottleneck ResNets under "
                                  "alpha 1 / beta 0 ('mixed': alpha 1 / beta 0 on both)")
    with torch.no_grad():
        x = sample.detach()
        if use_tc:
            # forward ONCE per call (the reference does the same, :70) + one contraction per layer per request
            eng = tcp.engine(precision, params)
            est = eng.forward(x)
            fh, fw = est.feat_hw
            want = (x.shape[0], est.feat_c, fh, fw)
            if tuple(target.shape) != want:
                raise RuntimeError(f"Mismatch in shape: grad_output[0] has a shape of {tuple(target.shape)} and "
                                   f"output[0] has a shape of {want}.")
            r_pix = target.detach().float().flatten(2).transpose(1, 2).contiguous()
            R = eng.relevance(est, r_pix)
            logits = eng.features(est, "nchw") if return_output else None
        else:
            logits = model._lrpx_plan.forward(x)
            if tuple(target.shape) != tuple(logits.shape):
                raise RuntimeError(f"Mismatch in shape: grad_output[0] has a shape of {tuple(target.shape)} and "
                                   f"output[0] has a shape of {tuple(logits.shape)}.")
            R = model._lrpx_plan.backward(target.detach().float(), conservation_trace)
    if os.environ.get("LRPX_NO_GRAD_ACCUMULATION", "0") == "1":
        output = R
    else:
        if sample.is_leaf and not sample.requires_grad:
            sample.requires_grad = True
        if sample.grad is None:
            sample.grad = R.clone()
        else:
            sample.grad += R
        assert sample.grad.sum() != 0
        output = sample.grad.clone().detach()
    if return_output:
        return output, logits
    return output


# ------------------------------------------------------------------------------------------------ gradient family (f4)
def encoder_gradient_simt(model, sample, target, guided=False, return_output=False):
    """The encoder half of the gradient-family explainers on the fp32 CUDA-core kernels: the input gradient of a
    conv / ReLU / max-pool Sequential for the output gradient ``target`` (ExplainGridTDGradient.explain_cnn, reference
    models/gridTDmodel.py:1510-1523, where autograd does it), or its guided-backpropagation variant (``guided``: every
    ReLU passes only the positive part of the incoming gradient where its output is positive, :1677-1723).
        conv     : W^T * g            = lrpx_conv_rule_rin_f32 in its PLAIN form against a tensor of ones
        ReLU     : g (.) [out > 0]    = lrpx_relu_mask_f32  (guided: of the clamped g)
        max-pool : g to the argmax    = lrpx_maxpool_wta_f32 (a window whose maximum is 0 gets 0: the ReLU below would
                                        zero it anyway)
    The precision='simt' path of the gradient explainers; the tensor-core chain (lrpx.tc, rule 'gradient' / 'guided') is
    the fast one."""
    if not sample.is_cuda:
        raise RuntimeError("lrpx: encoder_gradient_simt needs a CUDA tensor (there is no CPU fallback)")
    if _is_bottleneck_resnet(model):
        return _resnet_gradient_simt(model, sample, target, guided, return_output)
    if not isinstance(model, nn.Sequential):
        raise NotImplementedError("the gradient explainers cover Sequential conv / ReLU / max-pool encoders and the "
                                  "Bottleneck ResNet of models/resnet.py")
    leaves = _flatten_sequential(model)
    for i, m in enumerate(leaves):
        if not isinstance(m, (nn.Conv2d, nn.ReLU, nn.MaxPool2d)):
            raise NotImplementedError(f"gradient explainers: unsupported layer {type(m)}")
        if isinstance(m, nn.MaxPool2d) and (i == 0 or not isinstance(leaves[i - 1], nn.ReLU)):
            raise NotImplementedError("gradient explainers: a max-pool must follow a ReLU")
    with torch.no_grad():
        x = sample.detach().float()
        outs = []
        for m in leaves:
            x = _leaf_forward(m, x)
            outs.append(x)
        if tuple(target.shape) != tuple(x.shape):
            raise RuntimeError(f"Mismatch in shape: grad_output[0] has a shape of {tuple(target.shape)} and "
                               f"output[0] has a shape of {tuple(x.shape)}.")
        g = target.detach().float().contiguous()
        for m, out in zip(reversed(leaves), reversed(outs)):
            a = m.input[0]
            if isinstance(m, nn.Conv2d):
                g = ops.conv_rule_rin(torch.ones_like(a), m.weight.detach(), g, m.stride, m.padding, m.dilation,
                                      net=ops.NET_PLAIN)
            elif isinstance(m, nn.ReLU):
                if guided:
                    g = ops.relu_mask(g, g)            # clamp(g, min=0)
                g = ops.relu_mask(out, g)
            else:
                g = ops.maxpool_wta(a, g, m.kernel_size, m.stride, m.padding)
    return (g, x) if return_output else g


def _resnet_gradient_simt(model, sample, target, guided=False, return_output=False):
    """encoder_gradient_simt for the Bottleneck ResNet of models/resnet.py (eval mode): convolutions of any stride through
    lrpx_conv_rule_rin_f32 (PLAIN, against ones), BatchNorm as its per-channel scale, ReLU masks, the overlapping 3x3/s2
    max-pool through lrpx_maxpool_wta_f32, the residual Add as a copy into both branches whose gradients meet again at
    the block input.  ``guided``: the reference hooks only the ReLUs that are direct children of the encoder
    (gridTDmodel.py:1687-1691: ``named_children``), i.e. the stem's; the ReLUs inside the blocks keep their plain
    derivative."""
    m = model
    if m.training:
        raise NotImplementedError("the gradient explainers need eval() mode (BatchNorm running statistics)")
    blocks = [b for L in (m.layer1, m.layer2, m.layer3, m.layer4) for b in L]
    conv = lambda c, x: ops.conv_forward(x, c.weight.detach(), None if c.bias is None else c.bias.detach(), c.stride,
                                         c.padding, c.dilation)
    scale = lambda bn: (bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().view(1, -1, 1, 1)
    bnf = lambda bn, x: x * scale(bn) + (bn.bias - bn.running_mean * bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().view(1, -1, 1, 1)
    dconv = lambda c, x_in, g: ops.conv_rule_rin(torch.ones_like(x_in), c.weight.detach(), g.contiguous(), c.stride, c.padding,
                                                 c.dilation, net=ops.NET_PLAIN)
    with torch.no_grad():
        x0 = sample.detach().float()
        r1 = torch.relu(bnf(m.bn1, conv(m.conv1, x0)))
        x = ops.maxpool_forward(r1, m.maxpool.kernel_size, m.maxpool.stride, m.maxpool.padding, return_indices=False)
        saved = []
        for b in blocks:
            o1 = torch.relu(bnf(b.bn1, conv(b.conv1, x)))
            o2 = torch.relu(bnf(b.bn2, conv(b.conv2, o1)))
            o3 = bnf(b.bn3, conv(b.conv3, o2))
            idn = x if b.downsample is None else bnf(b.downsample[1], conv(b.downsample[0], x))
            out = torch.relu(o3 + idn)
            saved.append((x, o1, o2, out))
            x = out
        if tuple(target.shape) != tuple(x.shape):
            raise RuntimeError(f"Mismatch in shape: grad_output[0] has a shape of {tuple(target.shape)} and "
                               f"output[0] has a shape of {tuple(x.shape)}.")
        g = target.detach().float().contiguous()
        for b, (x_in, o1, o2, out) in zip(reversed(blocks), reversed(saved)):
            g = ops.relu_mask(out, g)
            go = dconv(b.conv3, o2, g * scale(b.bn3))
            go = dconv(b.conv2, o1, ops.relu_mask(o2, go) * scale(b.bn2))
            go = dconv(b.conv1, x_in, ops.relu_mask(o1, go) * scale(b.bn1))
            gi = g if b.downsample is None else dconv(b.downsample[0], x_in, g * scale(b.downsample[1]))
            g = go + gi
        g = ops.maxpool_wta(r1, g, m.maxpool.kernel_size, m.maxpool.stride, m.maxpool.padding)
        if guided:
            g = ops.relu_mask(g, g)
        g = dconv(m.conv1, x0, ops.relu_mask(r1, g) * scale(m.bn1))
    return (g, x) if return_output else g
