"""Shared host logic of the gradient-family explainers (SURVEY.md §8 f4): the reference's ExplainGridTDGradient /
ExplainiGridTDGuidedGradient / ExplainGridTDGradCam / ExplainGridTDGuidedGradCam (models/gridTDmodel.py:1214-1859) and
their AoA twins (models/aoamodel.py:1257-1776).

The reference pairs a hand-written, per-vector backward pass of the decoder (attention weights and gates held constant)
with torch autograd through a deep copy of the CNN, once per word.  Here a caption is ONE batched decoder-gradient call
(``lrpx_gridtd_decoder_grad_f32`` / ``lrpx_aoa_decoder_grad_f32``) and ONE batched pass of the tcgen05 chain in its
'gradient' / 'guided' rule (``lrpx.tc.TcVggEngine``: full weights W^T, gain = the ReLU's derivative, the max-pool
scatter; 'guided' clamps the gradient at every ReLU like the reference's backward hooks).  ``precision``: 'fp32'
(default; error-compensated bf16x3 operands), 'bf16', or 'simt' (fp32 CUDA-core kernels, ``encoder_gradient_simt``).
"""
import numpy as np
import torch

from LRPtools import lrp_wrapper
from lrpx import ops


def gridtd_grad_weights(sd):
    """B operands of lrpx_gridtd_grad_args from a GridTDModel state_dict."""
    H = sd["fc.weight"].shape[1]
    return {
        "W1": sd["AdaLSTM.lstm_cell.weight_ih"].contiguous(),                                           # (4H, H+2E)
        "W2": torch.cat((sd["LanguageLSTM.weight_ih"], sd["LanguageLSTM.weight_hh"]), 1).contiguous(),  # (4H, 3H)
        "W_fc": sd["fc.weight"].contiguous(),
        "W_glob": sd["global_img_feature_proj.weight"].contiguous(),
        "W_proj": sd["img_projector.weight"].reshape(H, -1).contiguous(),
    }


def aoa_grad_weights(sd):
    """B operands of lrpx_aoa_grad_args from an AOAModel state_dict."""
    H = sd["fc.weight"].shape[1]
    return {
        "W_g": torch.cat((sd["LanguageLSTM.weight_ih"], sd["LanguageLSTM.weight_hh"]), 1).contiguous(),  # (4H, E+2H)
        "W_fc": sd["fc.weight"].contiguous(),
        "W_aoa": sd["decoder_aoa_linear.weight"].contiguous(),
        "W_gate": sd["decoder_aoa_linear_gate.weight"].contiguous(),
        "W_v": sd["decoder_v_proj.weight"].contiguous(),
        "W_proj": sd["img_projector.weight"].reshape(H, -1).contiguous(),
    }


# ------------------------------------------------------------------------------------------ pyramid_expand as an operator
def _mirror(i, n):
    """index reflection about the edge pixel centres (d c b | a b c d | c b a): skimage's warp mode 'reflect'"""
    if n == 1:
        return 0
    period = 2 * (n - 1)
    i = abs(i) % period
    return period - i if i >= n else i


def _half_sample(i, n):
    """index reflection about the array edge (d c b a | a b c d | d c b a): scipy.ndimage's mode 'reflect'"""
    period = 2 * n
    i = i % period
    return period - 1 - i if i >= n else i


def expand_operator(n_in, upscale=16, sigma=None, truncate=4.0):
    """skimage.transform.pyramid_expand(order=1, mode='reflect') along one axis as a (n_in*upscale, n_in) matrix:
    bilinear resize (pixel centres at +0.5, mirror at the border) followed by scipy's Gaussian filter (sigma =
    2*upscale/6, radius int(truncate*sigma + 0.5), half-sample-symmetric border).  Both steps are separable, so the 2-D
    expansion of a (h, w) map M is  K_h M K_w^T.  skimage is not installed in this image: the operator follows the
    library's published definition ("parity unpinned", DESIGN.md §0)."""
    n_out = int(np.ceil(upscale * n_in))
    U = np.zeros((n_out, n_in))
    for r in range(n_out):
        src = (r + 0.5) / upscale - 0.5
        lo = int(np.floor(src))
        d = src - lo
        U[r, _mirror(lo, n_in)] += 1.0 - d
        U[r, _mirror(lo + 1, n_in)] += d
    sigma = 2 * upscale / 6.0 if sigma is None else sigma
    radius = int(truncate * sigma + 0.5)
    k = np.exp(-0.5 * (np.arange(-radius, radius + 1) / sigma) ** 2)
    k /= k.sum()
    G = np.zeros((n_out, n_out))
    for r in range(n_out):
        for j, wgt in enumerate(k):
            G[r, _half_sample(r + j - radius, n_out)] += wgt
    return G @ U


class GradientFamily:
    """Mixin in front of ExplainGridTDAttention / ExplainAOAAttention (whose encoder plumbing, caption search and
    explainer forward it reuses)."""
    RULE = "gradient"            # encoder rule of the tcgen05 chain: 'gradient' | 'guided'
    GUIDED_DECODER = False       # gridTD guided variants: d_img_feature[image_features <= 0] = 0 (gridTDmodel.py:1674)
    CAM = None                   # None | 'cam' (Grad-CAM map instead of the image gradient) | 'guided' (guided x CAM)
    ACCUMULATE_LIKE_REFERENCE = False     # the gradient explain_cnn works on a fresh copy of the image every time
    GRADIENT = True

    def _grad_weights(self):
        """The decoder-gradient kernels' weights (``_GRAD_WEIGHTS(state_dict)``), rebuilt when a model parameter is
        replaced or updated in place; the dict stays the same object until then."""
        return self._caches["grad"].get(self.model.parameters(), lambda: self._GRAD_WEIGHTS(self._state_dict()))

    def _check_encoder(self):
        # Bottleneck ResNets: the fp32 CUDA-core path only (LRPtools.lrp_wrapper.encoder_gradient_simt), except for Grad-CAM,
        # which needs the encoder's forward and no gradient chain (the tensor-core forward of lrpx.tc_resnet)
        if getattr(self, "is_resnet", False) and self.precision in ("bf16", "mixed") and self.CAM != "cam":
            raise NotImplementedError(f"precision={self.precision!r}: on a ResNet encoder the gradient-family explainers "
                                      "support precision 'fp32' and 'simt' (the fp32 CUDA-core kernels)")

    def explainer_forward(self, feat, tokens, quirk_double_bias_ih=False, want_gates=True):
        # the gradient explainers' LSTM forwards add bias_ih + bias_hh (gridTDmodel.py:1265): no Q3 here
        return super().explainer_forward(feat, tokens, quirk_double_bias_ih=False, want_gates=True)

    # ------------------------------------------------------------------ encoder half
    def _pix(self, d_img_feature):
        return d_img_feature.flatten(2).transpose(1, 2).contiguous()

    def _encoder_gradient(self, d_pix, rows):
        """d_pix (Q,P,C) gradient of the encoder output -> (Q,3,H,W) image gradient in this class's rule"""
        if self.uses_tc:
            return self.engine().relevance(self._enc_state, d_pix, rows)
        enc = self.model.img_encoder.encoder
        fh, fw = self._feat_hw
        guided = self.RULE == "guided"
        return torch.cat([lrp_wrapper.encoder_gradient_simt(enc, self.img, d_pix[q].t().reshape(1, -1, fh, fw), guided)
                          for q in range(d_pix.shape[0])])

    def _cam(self, d_pix, rows):
        return ops.grad_cam(self._state["feat"], d_pix, rows)

    def grad_cam(self, img_feature, grads):
        """reference gridTDmodel.py:1760-1771 / :1799-1810 on (1, C, h, w) tensors: the (h*w,) map of the Grad-CAM
        classes, the (h, w) map of the guided Grad-CAM ones (``lrpx_grad_cam_f32``)."""
        cam = ops.grad_cam(self._pix(img_feature), self._pix(grads))[0]
        return cam.view(img_feature.shape[2], img_feature.shape[3]) if self.CAM == "guided" else cam

    def _expand_ops(self, fh, fw, H, W):
        """(Kh (H, fh), Kw (W, fw)): pyramid_expand of an (fh, fw) Grad-CAM map to an (H, W) image as two operators, built
        once per size"""
        key = (fh, fw, H, W)
        if getattr(self, "_expand_key", None) != key:
            up = H // fh
            if (fh * up, fw * up) != (H, W):
                raise NotImplementedError("guided Grad-CAM needs an image size that is a multiple of the feature map's")
            to = lambda a: torch.tensor(a, dtype=torch.float32, device=self.device)
            self._expand = (to(expand_operator(fh, up)), to(expand_operator(fw, up)))
            self._expand_key = key
        return self._expand

    def _finish(self, d_pix, rows):
        """what explain_cnn returns for every request of d_pix"""
        if self.CAM == "cam":
            return self._cam(d_pix, rows)                                  # (Q, P)
        g = self._encoder_gradient(d_pix, rows)
        if self.CAM == "guided":
            fh, fw = self._feat_hw
            Kh, Kw = self._expand_ops(fh, fw, self.img.shape[2], self.img.shape[3])
            g = ops.cam_expand_mul(g, self._cam(d_pix, rows).view(-1, fh, fw), Kh, Kw)
        return g

    def explain_cnn(self, d_img_feature):
        """reference gridTDmodel.py:1510-1523 (gradient), :1702-1723 (guided), :1755-1758 (Grad-CAM -> (1, P)),
        :1812-1833 (guided Grad-CAM)."""
        rows = torch.zeros(d_img_feature.shape[0], dtype=torch.int32, device=self.device)
        return self._finish(self._pix(d_img_feature), rows)

    def _explain_image(self, d_feat):
        return self._finish(d_feat, torch.zeros(d_feat.shape[0], dtype=torch.int32, device=self.device))
