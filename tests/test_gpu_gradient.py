"""GPU parity of the gradient-family explainers (SURVEY.md §8 f4): the batched decoder-gradient kernels, Grad-CAM, the
'gradient' / 'guided' rules of the tcgen05 chain and the mirrors of the reference's Explain*Gradient / *GuidedGradient /
*GradCam / *GuidedGradCam classes — against fixtures the reference itself produced (gridtd_grad_512, aoa_grad_512,
gradient_e2e) and against the oracle on ragged multi-image batches."""
import argparse

import numpy as np
import pytest
import torch

import helpers
import lrp_oracle as O
import synth
from conftest import assert_close, spearman

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _pix(r):
    """(1,C,h,w) -> (P,C) pixel-major"""
    return r[0].reshape(r.shape[1], -1).t()


def _rel_l2(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / b.norm())


def _args(E, H, tmp_path):
    return argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")


@pytest.mark.parametrize("tc_gemm", [False, True])
def test_gridtd_decoder_grad_vs_reference_fixture(golden, tmp_path, tc_gemm):
    """Explainer forward (fused kernels, incl. the extra gates) + lrpx_gridtd_decoder_grad_f32 vs the reference's own
    ExplainGridTDGradient / ExplainiGridTDGuidedGradient / ExplainGridTDGradCam at the benched decoder size.
    fp32 CUDA-core GEMMs: scale-relative 1e-5; bf16x3 tensor-core GEMMs: 1e-4."""
    from lrpx import ops
    from models import gridTDmodel as G
    g = golden("gridtd_grad_512")
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(int(g["seed"]), V, H, E), strict=False)
    model.to(DEV).eval()
    ex = G.ExplainGridTDGradient(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="simt")
    toks = g["tokens"].tolist()
    feat = _pix(g["feats"]).unsqueeze(0).to(DEV).contiguous()
    st = ex.explainer_forward(feat, torch.tensor([toks], device=DEV))
    assert_close(st["pred"][0], g["predictions"], rtol=1e-4, atol=2e-5, what="predictions")
    for k, ref in (("o1", "o1"), ("o2", "o2"), ("sg", "sen_gate")):
        assert_close(st[k][0], g[ref], rtol=1e-4, atol=2e-6, what=k)
    ts = g["ts"].tolist()
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=DEV)
    atol = 1e-4 if tc_gemm else 1e-5
    for key, guided in (("grad", False), ("guided", True)):
        d_feat, r_words = ops.gridtd_decoder_grad(st, ex._grad_weights(), i32([0] * len(ts)), i32(ts),
                                                  i32([toks[t + 1] for t in ts]), guided=guided, tc_gemm=tc_gemm)
        for q, t in enumerate(ts):
            ref = _pix(g[f"{key}_d_feat_{t}"])
            scale = ref.abs().max()
            print(f"gridTD {key} tc_gemm={tc_gemm} t={t}: max scale-relative error "
                  f"{float((d_feat[q].cpu() - ref).abs().max() / scale):.3e}")
            assert_close(d_feat[q] / scale, ref / scale, rtol=1e-4, atol=atol, what=f"{key} d_feat t={t}")
            assert_close(r_words[q, :t + 1], g[f"{key}_r_words_{t}"], rtol=1e-4, atol=atol, what=f"{key} r_words t={t}")
            assert float(r_words[q, t + 1:].abs().sum()) == 0.0
            if not guided:
                cam = ops.grad_cam(feat, d_feat[q:q + 1])
                assert_close(cam[0], g[f"cam_{t}"].reshape(-1), rtol=1e-3, atol=10 * atol, what=f"cam t={t}")


@pytest.mark.parametrize("tc_gemm", [False, True])
def test_aoa_decoder_grad_vs_reference_fixture(golden, tmp_path, tc_gemm):
    from lrpx import ops
    from models import aoamodel as A
    g = golden("aoa_grad_512")
    V, H, E, C = int(g["V"]), int(g["H"]), int(g["E"]), int(g["C"])
    model = A.AOAModel(E, H, 8, V, "vgg16")
    model.load_state_dict(synth.aoa_decoder_state(int(g["seed"]), V, H, E, C), strict=False)
    model.to(DEV).eval()
    ex = A.ExplainAOAGradient(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="simt")
    toks = g["tokens"].tolist()
    feat = _pix(g["feats"]).unsqueeze(0).to(DEV).contiguous()
    st = ex.explainer_forward(feat, torch.tensor([toks], device=DEV))
    assert_close(st["pred"][0], g["predictions"], rtol=1e-4, atol=2e-5, what="predictions")
    assert_close(st["o"][0], g["ot"], rtol=1e-4, atol=2e-6, what="output gate")
    assert_close(st["caoa_gate"][0], g["context_aoa_gate"], rtol=1e-4, atol=2e-5, what="aoa gate")
    cases = g["cases"].tolist()
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=DEV)
    d_feat, r_words = ops.aoa_decoder_grad(st, ex._grad_weights(), 8, i32([0] * len(cases)), i32([t for t, _ in cases]),
                                           i32([toks[t + 1] for t, _ in cases]), i32([h for _, h in cases]), tc_gemm=tc_gemm)
    atol = 1e-4 if tc_gemm else 1e-5
    for q, (t, hd) in enumerate(cases):
        ref = _pix(g[f"d_feat_{t}_{hd}"])
        scale = ref.abs().max()
        print(f"AoA tc_gemm={tc_gemm} t={t} head={hd}: max scale-relative error "
              f"{float((d_feat[q].cpu() - ref).abs().max() / scale):.3e}")
        assert_close(d_feat[q] / scale, ref / scale, rtol=1e-4, atol=atol, what=f"d_feat {t},{hd}")
        assert_close(r_words[q, :t + 1], g[f"r_words_{t}_{hd}"], rtol=1e-4, atol=atol, what=f"r_words {t},{hd}")
        cam = ops.grad_cam(feat, d_feat[q:q + 1])
        assert_close(cam[0], g[f"cam_{t}_{hd}"].reshape(-1), rtol=1e-3, atol=10 * atol, what=f"cam {t},{hd}")
    # the named helper (reference :1415-1433)
    dv = ex.gradient_mha(torch.arange(H, device=DEV, dtype=torch.float32), st["alpha"][0, 2], 3)
    assert dv.shape == (st["alpha"].shape[-1], H) and float(dv[:, :3 * 64].abs().sum()) == 0.0
    assert_close(dv[:, 3 * 64:4 * 64], st["alpha"][0, 2, 3].unsqueeze(1) * torch.arange(192, 256, device=DEV).float(), what="gradient_mha")


def test_decoder_grad_batched_ragged_vs_oracle():
    """several images, ragged captions, requests in arbitrary order incl. duplicates and t = 0; both decoders"""
    from lrpx import ops
    from models._gradient import gridtd_grad_weights, aoa_grad_weights
    V, H, E = 120, 64, 32
    p = synth.gridtd_decoder_state(7, V, H, E, C=64, n_pixel=16)
    pa = synth.aoa_decoder_state(8, V, H, E, C=64)
    gs, as_, toks = [], [], []
    for b, T in enumerate([5, 3, 1]):
        f = torch.randn(64, 4, 4, generator=torch.Generator().manual_seed(100 + b)).clamp(min=0)
        tk = synth.tokens(200 + b, T, V)
        toks.append(tk)
        gs.append(O.gridtd_explainer_forward(p, f, tk, gradient=True))
        as_.append(O.aoa_explainer_forward(pa, f, tk, 8, gradient=True))
    reqs = [(0, 4), (1, 0), (2, 0), (0, 0), (1, 2), (0, 4), (0, 2)]
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=DEV)
    req_img, req_t = i32([b for b, _ in reqs]), i32([t for _, t in reqs])
    req_word = i32([toks[b][t + 1] for b, t in reqs])
    ks = helpers.gridtd_grad_kernel_state(gs, DEV)
    W = helpers.to_dev(gridtd_grad_weights(p), DEV)
    for guided in (False, True):
        d_feat, r_words = ops.gridtd_decoder_grad(ks, W, req_img, req_t, req_word, guided=guided)
        for q, (b, t) in enumerate(reqs):
            df, rw = O.gridtd_gradient_wordt(p, gs[b], t, guided=guided)
            scale = df.abs().max()
            assert_close(d_feat[q] / scale, df / scale, rtol=1e-4, atol=1e-5, what=f"gridTD guided={guided} request {q}")
            assert_close(r_words[q, :t + 1], rw, rtol=1e-4, atol=1e-5, what=f"gridTD r_words request {q}")
    ka = helpers.aoa_grad_kernel_state(as_, DEV)
    Wa = helpers.to_dev(aoa_grad_weights(pa), DEV)
    heads = [q % 8 for q in range(len(reqs))]
    d_feat, r_words = ops.aoa_decoder_grad(ka, Wa, 8, req_img, req_t, req_word, i32(heads))
    for q, (b, t) in enumerate(reqs):
        df, rw = O.aoa_gradient_wordt(pa, as_[b], t, heads[q])
        scale = df.abs().max()
        assert_close(d_feat[q] / scale, df / scale, rtol=1e-4, atol=1e-5, what=f"AoA request {q}")
        assert_close(r_words[q, :t + 1], rw, rtol=1e-4, atol=1e-5, what=f"AoA r_words request {q}")


@pytest.mark.parametrize("guided", [False, True])
@pytest.mark.parametrize("precision", ["simt", "fp32", "bf16"])
def test_encoder_gradient_vs_oracle(precision, guided):
    """The image gradient / guided backpropagation through a VGG-style encoder at 64x64: the tcgen05 chain in its
    'gradient' / 'guided' rule (fp32-accurate and bf16 modes) and the fp32 CUDA-core path vs the oracle's layer-by-layer
    backward (= autograd; guided = the reference's ReLU hooks).  Two images, five requests."""
    import torch.nn as nn
    from LRPtools import lrp_wrapper
    from lrpx import tc
    cfg = [64, 64, "M", 128, 128, "M", 256, "M", 256]
    sd = synth.vgg_state(91, cfg)
    layers = O.vgg_layers_from_state(sd, cfg)
    x = synth.images(92, 2, 64)
    feat = O.sequential_forward(layers, x)[-1]                                  # (2,256,8,8)
    gen = torch.Generator().manual_seed(93)
    rows = [0, 1, 1, 0, 1]
    tgt = torch.randn(len(rows), *feat.shape[1:], generator=gen)
    want = torch.cat([O.sequential_gradient(layers, x[b:b + 1], tgt[q:q + 1], guided=guided) for q, b in enumerate(rows)])
    if precision == "simt":
        mods, idx = [], 0
        for v in cfg:
            if v == "M":
                mods.append(nn.MaxPool2d(2, 2)); idx += 1
            else:
                c = nn.Conv2d(sd[f"{idx}.weight"].shape[1], v, 3, padding=1)
                c.load_state_dict({"weight": sd[f"{idx}.weight"], "bias": sd[f"{idx}.bias"]})
                mods += [c, nn.ReLU(True)]; idx += 2
        enc = nn.Sequential(*mods).to(DEV)
        got = torch.cat([lrp_wrapper.encoder_gradient_simt(enc, x[b:b + 1].to(DEV), tgt[q:q + 1].to(DEV), guided)
                         for q, b in enumerate(rows)])
    else:
        ws = [sd[k] for k in sd if k.endswith("weight")]
        bs = [sd[k] for k in sd if k.endswith("bias")]
        rule = "guided" if guided else "gradient"
        eng = (tc.TcVggMixed(ws, bs, cfg, DEV, rule=rule) if precision == "bf16" else
               tc.TcVggEngine(ws, bs, cfg, DEV, precision=precision, rule=rule))
        st = eng.forward(x.to(DEV))
        assert_close(eng.features(st, "nchw"), feat, rtol=1e-4, atol=2e-5 * float(feat.abs().max()), what="features")
        got = eng.relevance(st, tgt.flatten(2).transpose(1, 2).contiguous().to(DEV), torch.tensor(rows, dtype=torch.int32, device=DEV))
    scale = want.abs().max()
    err = float((got.cpu() - want).abs().max() / scale)
    print(f"encoder gradient precision={precision} guided={guided}: max scale-relative error {err:.3e}, rel-L2 "
          f"{_rel_l2(got, want):.3e}, Spearman {spearman(got, want):.5f}")
    # A gradient is discontinuous in the forward pass: a ReLU whose pre-activation is within the forward's rounding
    # error of zero flips its mask and moves the ~600 input-gradient entries it feeds by ~4 % each.  The fp32 CUDA-core
    # forward (1e-7 relative) reproduces the oracle's masks; the error-compensated tensor-core forward (1e-5 relative,
    # one-sided by the round-toward-zero accumulation) flips ~2e-6 of the units per layer, the bf16 forward (4e-3) many
    # more — which is why precision 'bf16' of the gradient family keeps the fp32-accurate FORWARD and runs only the chain
    # in bf16 (measured: same error as the fp32-accurate chain).  Bars = 2x the measured figures (profiles/README.md):
    # guided backpropagation, which zeroes negative gradients at every ReLU, is an order of magnitude less sensitive
    # than the plain gradient.
    if precision == "simt":
        assert_close(got / scale, want / scale, rtol=1e-4, atol=1e-5, what="simt gradient")
    elif precision == "fp32":
        assert _rel_l2(got, want) < (3e-3 if guided else 3e-2) and spearman(got, want) > 0.999
    else:       # bf16 chain on the fp32-accurate forward's masks (TcVggMixed): the mask flips dominate, as above
        assert _rel_l2(got, want) < (5e-3 if guided else 4e-2) and spearman(got, want) > 0.999


@pytest.mark.parametrize("cls,key", [("ExplainGridTDGradient", "grad"), ("ExplainiGridTDGuidedGradient", "guided")])
@pytest.mark.parametrize("precision", ["fp32", "simt"])
def test_gradient_explainers_end_to_end_vs_reference_fixture(golden, tmp_path, cls, key, precision):
    """explain_caption of the mirrors vs the reference's own run (fixture gradient_e2e: seeded VGG16 at 224x224, small
    decoder, caption search capped at 7 words): same caption, heat-maps of the first and the last word, all word
    relevances.  Measured on B200 (rel-L2 of a heat-map): 'simt' (fp32 CUDA cores) 4e-3 plain / 2e-4 guided — fp32 on
    both sides, yet a few ReLU masks flip with the summation order; 'fp32' (the tcgen05 chain, fp32-accurate mode)
    1.5e-2 plain / 1.9e-3 guided, Spearman >= 0.9999."""
    from models import gridTDmodel as G
    g = golden("gradient_e2e")
    V, H, E, seed = int(g["V"]), int(g["H"]), int(g["E"]), int(g["seed"])
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(seed, V, H, E), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(seed + 1))
    model.to(DEV).eval()
    ex = getattr(G, cls)(_args(E, H, tmp_path), synth.word_map(V), model=model, precision=precision)
    img = synth.images(seed + 2, 1).to(DEV)
    ex.preprocess_img = lambda p: img
    find = ex._find_caption
    ex._find_caption = lambda path, beam_size, max_cap_length: find(path, beam_size, 7)
    imgs, words = ex.explain_caption("synthetic.jpg")
    toks = ex.beam_caption_encode
    assert toks == g["tokens"].tolist(), (toks, g["tokens"].tolist())
    T = len(toks) - 1
    assert_close(torch.cat(words), g[f"{key}_words"], rtol=1e-3, atol=1e-4, what="word relevances")
    for t in (0, T - 1):
        ref = g[f"{key}_img_{t}"]
        scale = ref.abs().max()
        err = float((imgs[t].cpu() - ref).abs().max() / scale)
        print(f"{cls} precision={precision} t={t}: max scale-relative error {err:.3e}, rel-L2 {_rel_l2(imgs[t], ref):.3e}, "
              f"Spearman {spearman(imgs[t], ref):.5f}")
        if precision == "simt":
            # fp32 on both sides, different summation order: a handful of ReLU masks flip in 13 layers (see
            # test_encoder_gradient_vs_oracle); everything else agrees to 2e-4 of the maximum
            off = ((imgs[t].cpu() - ref).abs() > 2e-4 * scale + 1e-3 * ref.abs()).float().mean()
            print(f"  fraction of elements beyond 2e-4 of the maximum: {float(off):.3e}")
            assert float(off) < (1e-2 if key == "guided" else 0.1) and _rel_l2(imgs[t], ref) < 1e-2, (t, float(off))
        else:
            assert _rel_l2(imgs[t], ref) < (2e-2 if key == "guided" else 0.2), (t, _rel_l2(imgs[t], ref))
    # explain_caption_wordt / explain_cnn, one word at a time, give the same as the batched call
    d_img, rw = ex.explain_caption_wordt(T - 1)
    one = ex.explain_cnn(d_img)
    assert_close(one, imgs[T - 1], rtol=1e-5, atol=1e-6 * float(imgs[T - 1].abs().max()), what="single-word path")


def test_gradcam_classes_and_guided_gradcam(golden, tmp_path):
    """ExplainGridTDGradCam.explain_cnn -> (1, P) map (checked against the oracle's grad_cam of the oracle's gradient);
    ExplainGridTDGuidedGradCam = guided backpropagation x the pyramid-expanded map (expansion operator checked against
    scipy in tests/test_models_cpu.py; skimage itself is absent: unpinned)."""
    from models import gridTDmodel as G
    from models._gradient import expand_operator
    g = golden("gradient_e2e")
    V, H, E, seed = int(g["V"]), int(g["H"]), int(g["E"]), int(g["seed"])
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(seed, V, H, E), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(seed + 1))
    model.to(DEV).eval()
    img = synth.images(seed + 2, 1).to(DEV)
    toks = g["tokens"].tolist()
    out = {}
    for cls in ("ExplainGridTDGradCam", "ExplainGridTDGuidedGradCam", "ExplainiGridTDGuidedGradient"):
        ex = getattr(G, cls)(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="fp32")
        ex.img = img
        ex.beam_caption_encode = toks
        ex._set_state(img, toks)
        t = len(toks) - 2
        d_img, _ = ex.explain_caption_wordt(t)
        out[cls] = (ex, d_img, ex.explain_cnn(d_img))
    ex, d_img, cam = out["ExplainGridTDGradCam"]
    assert cam.shape == (1, 196)
    want = O.grad_cam(ex._state["feat"][0].cpu(), _pix(d_img.cpu()))
    assert_close(cam[0], want, rtol=1e-3, atol=1e-5, what="Grad-CAM map")
    ex2, d_img2, ggc = out["ExplainGridTDGuidedGradCam"]
    guided = out["ExplainiGridTDGuidedGradient"][2]
    cam2 = O.grad_cam(ex2._state["feat"][0].cpu(), _pix(d_img2.cpu())).reshape(14, 14).double()
    K = torch.tensor(expand_operator(14, 16))
    up = (K @ cam2 @ K.t()).float()
    assert_close(ggc.cpu(), guided.cpu() * up, rtol=1e-4, atol=1e-6 * float(guided.abs().max()), what="guided Grad-CAM")


@pytest.mark.parametrize("cls,guided", [("ExplainAOAGradient", False), ("ExplainAOAGuidedGradient", True)])
def test_aoa_gradient_explainers_end_to_end_vs_oracle(tmp_path, cls, guided):
    """ExplainAOAGradient / ExplainAOAGuidedGradient.explain_caption(img, head) through a seeded VGG-style encoder at 64x64
    (fp32 CUDA-core path, so that the ReLU masks are the oracle's): caption from the mirror's own search, decoder gradient
    + encoder backward of the oracle on that caption."""
    import torch.nn as nn
    from models import aoamodel as A
    V, H, E, head = 80, 64, 32, 5
    model = A.AOAModel(E, H, 8, V, "vgg16")
    dec = synth.aoa_decoder_state(301, V, H, E, 512)
    model.load_state_dict(dec, strict=False)
    vs = synth.vgg_state(302)
    model.img_encoder.encoder.load_state_dict(vs)
    model.to(DEV).eval()
    ex = getattr(A, cls)(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="simt")
    img = synth.images(303, 1, 64)
    ex.preprocess_img = lambda p: img.to(DEV)
    find = ex._find_caption
    ex._find_caption = lambda path, beam_size, max_cap_length: find(path, beam_size, 6)
    imgs, words = ex.explain_caption("synthetic.jpg", head)
    toks = ex.beam_caption_encode
    T = len(toks) - 1
    assert T >= 1 and len(imgs) == T and imgs[0].shape == (1, 3, 64, 64)
    layers = O.vgg_layers_from_state(vs)
    feat = O.sequential_forward(layers, img)[-1]
    st = O.aoa_explainer_forward(dec, feat[0], toks, 8, gradient=True)
    assert_close(ex.predictions, st["pred"], rtol=1e-3, atol=1e-4, what="predictions")
    for t in range(T):
        df, rw = O.aoa_gradient_wordt(dec, st, t, head)
        want = O.sequential_gradient(layers, img, df.t().reshape(1, -1, *feat.shape[-2:]), guided=guided)
        scale = want.abs().max()
        assert _rel_l2(imgs[t], want) < 5e-3, (t, _rel_l2(imgs[t], want))
        off = ((imgs[t].cpu() - want).abs() > 2e-4 * scale + 1e-3 * want.abs()).float().mean()
        assert float(off) < 5e-2, (t, float(off))
        assert_close(words[t], rw, rtol=1e-3, atol=1e-5, what=f"r_words t={t}")


@pytest.mark.parametrize("cls", ["ExplainGridTDGradient", "ExplainiGridTDGuidedGradient"])
def test_batch_explainer_with_gradient_explainers(tmp_path, cls):
    """lrpx.pipeline.BatchExplainer drives the gradient-family explainers like the relevance ones: 2 images x 4 words in
    one pass (eager and CUDA-graph replay) = the per-image explain_caption_wordt / explain_cnn results."""
    from models import gridTDmodel as G
    from lrpx.pipeline import BatchExplainer
    V, H, E, T = 60, 64, 32, 4
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(311, V, H, E), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(312))
    model.to(DEV).eval()
    ex = getattr(G, cls)(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="fp32")
    imgs = synth.images(313, 2).to(DEV)
    toks = torch.tensor([synth.tokens(314, T, V), synth.tokens(315, T, V)], device=DEV)
    # tc_gemm=False: the decoder GEMMs on fp32 CUDA cores, as the one-word path of precision 'fp32' runs them
    heat, r_words = BatchExplainer(ex, chunk=4, tc_gemm=False).explain(imgs, toks)
    heat = heat.clone()
    heat_g, words_g = BatchExplainer(ex, chunk=4, use_graph=True, tc_gemm=False).explain(imgs, toks)
    assert_close(heat_g, heat, rtol=0, atol=0, what="graph replay")
    assert_close(words_g, r_words, rtol=0, atol=0, what="graph replay words")
    for b in range(2):
        ex.img = imgs[b:b + 1]
        ex.beam_caption_encode = toks[b].tolist()
        ex._set_state(ex.img, ex.beam_caption_encode)
        for t in (0, T - 1):
            d_img, rw = ex.explain_caption_wordt(t)
            one = ex.explain_cnn(d_img)
            q = b * T + t
            # the explainer forward's library GEMMs pick another algorithm for 2 rows than for 1: ~1e-5 of the maximum
            assert_close(heat[q:q + 1], one, rtol=1e-3, atol=1e-4 * float(one.abs().max()), what=f"image {b} word {t}")
            assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=1e-5, what=f"words image {b} word {t}")


@pytest.mark.parametrize("guided", [False, True])
def test_resnet_encoder_gradient_vs_autograd(guided):
    """Gradient explainers on a Bottleneck ResNet encoder (fp32 CUDA-core path): input gradient vs torch autograd through
    the same module (eval mode), 64x64 image, blocks [2, 1, 1, 1]; guided = the reference's hooks, which reach only the
    stem's ReLU of a ResNet (named_children of the encoder, gridTDmodel.py:1687-1691)."""
    import models.resnet as R
    from LRPtools import lrp_wrapper
    torch.manual_seed(17)
    net = R.ResNet(R.Bottleneck, [2, 1, 1, 1])
    g = torch.Generator().manual_seed(18)
    for m in net.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.2)
            m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
            m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.2)
    enc = torch.nn.Sequential(*list(net.children())[:-2]).to(DEV).eval()
    body = enc                     # conv1, bn1, relu, maxpool, layer1..4
    x = synth.images(19, 1, 64).to(DEV)
    xr = x.clone().requires_grad_(True)
    handles = []
    if guided:
        relu = body[2]
        relu.inplace = False
        handles.append(relu.register_full_backward_hook(lambda mod, gi, go: (go[0].clamp(min=0) * (mod._out > 0).float(),)))
        handles.append(relu.register_forward_hook(lambda mod, i, o: setattr(mod, "_out", o.detach())))
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False          # the autograd side in true fp32 (cuDNN's default would be TF32)
    try:
        feat = body(xr)
        tgt = torch.randn(feat.shape, generator=torch.Generator().manual_seed(20)).to(DEV)
        feat.backward(tgt)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    want = xr.grad.detach()
    for h in handles:
        h.remove()
    # the plan walks the ResNet object: rebuild one that shares the Sequential's modules
    res = R.ResNet(R.Bottleneck, [2, 1, 1, 1])
    res.conv1, res.bn1, res.relu, res.maxpool, res.layer1, res.layer2, res.layer3, res.layer4 = list(body.children())
    res.to(DEV).eval()
    got, f2 = lrp_wrapper.encoder_gradient_simt(res, x, tgt, guided=guided, return_output=True)
    assert_close(f2, feat.detach(), rtol=1e-3, atol=1e-4 * float(feat.detach().abs().max()), what="features")
    print(f"ResNet gradient guided={guided}: rel-L2 {_rel_l2(got, want):.3e}, Spearman {spearman(got, want):.6f}")
    assert _rel_l2(got, want) < 1e-2 and spearman(got, want) > 0.999


def test_gradient_explainer_with_resnet101_encoder(tmp_path):
    """ExplainGridTDGradient on a ResNet101 encoder (7x7 grid of 2048-d features): the encoder half runs on the fp32
    CUDA-core path; explain_cnn of the word's decoder gradient = torch autograd through the same encoder."""
    from models import gridTDmodel as G
    V, H, E = 60, 64, 32
    torch.manual_seed(23)
    model = G.GridTDModel(E, H, V, "resnet101", n_pixel=49)
    model.load_state_dict(synth.gridtd_decoder_state(331, V, H, E, C=2048, n_pixel=49), strict=False)
    model.to(DEV).eval()
    args = _args(E, H, tmp_path)
    args.encoder = "resnet101"
    ex = G.ExplainGridTDGradient(args, synth.word_map(V), model=model)
    assert not ex.uses_tc and ex.is_resnet
    with pytest.raises(NotImplementedError):
        G.ExplainGridTDGradient(args, synth.word_map(V), model=model, precision="bf16")
    img = synth.images(332, 1).to(DEV)
    toks = synth.tokens(333, 2, V)
    ex.preprocess_img = lambda p: img
    model.beam_search = lambda *a, **k: (["a b"], toks[1:])
    heat, words = ex.explain_caption("synthetic.jpg")
    assert len(heat) == 2 and heat[0].shape == (1, 3, 224, 224) and words[1].shape == (2,)
    d_img, _ = ex.explain_caption_wordt(1)
    assert d_img.shape == (1, 2048, 7, 7)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        xr = img.clone().requires_grad_(True)
        model.img_encoder.encoder(xr).backward(d_img)
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    assert _rel_l2(heat[1], xr.grad) < 2e-2 and spearman(heat[1], xr.grad) > 0.999, _rel_l2(heat[1], xr.grad)


def test_decoder_grad_long_caption_wide_state_vs_oracle():
    """T x (P + H) beyond one block's shared memory (45 steps, H = 1152): the per-(pixel, request) form of the attention
    accumulation takes over; same result as the oracle."""
    from lrpx import ops
    from models._gradient import gridtd_grad_weights
    V, H, E, T = 50, 1152, 64, 45
    p = synth.gridtd_decoder_state(41, V, H, E, C=64, n_pixel=16)
    f = torch.randn(64, 4, 4, generator=torch.Generator().manual_seed(42)).clamp(min=0)
    tk = synth.tokens(43, T, V)
    st = O.gridtd_explainer_forward(p, f, tk, gradient=True)
    ks = helpers.gridtd_grad_kernel_state([st], DEV)
    W = helpers.to_dev(gridtd_grad_weights(p), DEV)
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=DEV)
    ts = [T - 1, 7]
    for tc_gemm in (False, True):
        d_feat, r_words = ops.gridtd_decoder_grad(ks, W, i32([0, 0]), i32(ts), i32([tk[t + 1] for t in ts]), tc_gemm=tc_gemm)
        for q, t in enumerate(ts):
            df, rw = O.gridtd_gradient_wordt(p, st, t)
            scale = df.abs().max()
            assert_close(d_feat[q] / scale, df / scale, rtol=1e-3, atol=1e-4 if tc_gemm else 1e-5, what=f"d_feat t={t}")
            assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=1e-4 if tc_gemm else 1e-5, what=f"r_words t={t}")


@pytest.mark.parametrize("tc_gemm", [False, True])
def test_adaptive_decoder_grad_vs_reference_fixture(golden, tmp_path, tc_gemm):
    """ExplainAdaptiveGradient (single-LSTM adaptive attention): explainer forward incl. the extra gates and
    lrpx_adaptive_decoder_grad_f32 vs the reference's own outputs (fixture adaptive_grad_512)."""
    from lrpx import ops
    from models import adaptiveattention as AA
    g = golden("adaptive_grad_512")
    V, H = int(g["V"]), int(g["H"])
    model = AA.AdaptiveAttentionCaptioningModel(H, H, V, "vgg16")
    model.load_state_dict(synth.adaptive_decoder_state(int(g["seed"]), V, H, H), strict=False)
    model.to(DEV).eval()
    ex = AA.ExplainAdaptiveGradient(_args(H, H, tmp_path), synth.word_map(V), model=model, precision="simt")
    toks = g["tokens"].tolist()
    feat = _pix(g["feats"]).unsqueeze(0).to(DEV).contiguous()
    st = ex.explainer_forward(feat, torch.tensor([toks], device=DEV))
    assert_close(st["pred"][0], g["predictions"], rtol=1e-4, atol=2e-5, what="predictions")
    assert_close(st["o"][0], g["ot"], rtol=1e-4, atol=2e-6, what="output gate")
    assert_close(st["sg"][0], g["sen_gate"], rtol=1e-4, atol=2e-6, what="sentinel gate")
    ts = g["ts"].tolist()
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=DEV)
    d_feat, r_words = ops.adaptive_decoder_grad(st, ex._grad_weights(), i32([0] * len(ts)), i32(ts),
                                                i32([toks[t + 1] for t in ts]), tc_gemm=tc_gemm)
    atol = 1e-4 if tc_gemm else 1e-5
    for q, t in enumerate(ts):
        ref = _pix(g[f"grad_d_feat_{t}"])
        scale = ref.abs().max()
        print(f"adaptive tc_gemm={tc_gemm} t={t}: max scale-relative error {float((d_feat[q].cpu() - ref).abs().max() / scale):.3e}")
        assert_close(d_feat[q] / scale, ref / scale, rtol=1e-4, atol=atol, what=f"d_feat t={t}")
        assert_close(r_words[q, :t + 1], g[f"grad_r_words_{t}"], rtol=1e-4, atol=atol, what=f"r_words t={t}")
        assert float(r_words[q, t + 1:].abs().sum()) == 0.0
    t = ts[-1]
    assert_close(d_feat[-1] / scale, _pix(g[f"guided_d_feat_{t}"]) / scale, rtol=1e-4, atol=atol, what="guided = plain decoder half")


def test_adaptive_gradient_explainers_end_to_end_vs_oracle(tmp_path):
    """ExplainiAdaptiveGuidedGradient.explain_caption through a seeded VGG-style encoder at 64x64 (fp32 CUDA-core path) vs
    the oracle's decoder gradient + guided backward on the caption the mirror found."""
    from models import adaptiveattention as AA
    V, H = 80, 64
    model = AA.AdaptiveAttentionCaptioningModel(H, H, V, "vgg16", n_pixel=16)
    dec = synth.adaptive_decoder_state(341, V, H, H, 512, n_pixel=16)
    model.load_state_dict(dec, strict=False)
    vs = synth.vgg_state(342)
    model.img_encoder.encoder.load_state_dict(vs)
    model.to(DEV).eval()
    ex = AA.ExplainiAdaptiveGuidedGradient(_args(H, H, tmp_path), synth.word_map(V), model=model, precision="simt")
    img = synth.images(343, 1, 64)
    ex.preprocess_img = lambda p: img.to(DEV)
    find = ex._find_caption
    ex._find_caption = lambda path, beam_size, max_cap_length: find(path, beam_size, 5)
    imgs, words = ex.explain_caption("synthetic.jpg")
    toks = ex.beam_caption_encode
    T = len(toks) - 1
    assert T >= 1 and len(imgs) == T
    layers = O.vgg_layers_from_state(vs)
    feat = O.sequential_forward(layers, img)[-1]
    st = O.adaptive_explainer_forward(dec, feat[0], toks)
    for t in range(T):
        df, rw = O.adaptive_gradient_wordt(dec, st, t)
        want = O.sequential_gradient(layers, img, df.t().reshape(1, -1, *feat.shape[-2:]), guided=True)
        assert _rel_l2(imgs[t], want) < 5e-3, (t, _rel_l2(imgs[t], want))
        assert_close(words[t], rw, rtol=1e-3, atol=1e-5, what=f"r_words t={t}")


def test_forward_greedy_and_named_grad_cam(tmp_path):
    """forward_greedy (reference gridTDmodel.py:799-890: the beam-size-1 caption's saved state) and the named grad_cam
    method of the CAM classes (:1760-1771)."""
    from models import gridTDmodel as G
    V, H, E = 60, 64, 32
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(351, V, H, E), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(352))
    model.to(DEV).eval()
    ex = G.ExplainGridTDGradCam(_args(E, H, tmp_path), synth.word_map(V), model=model)
    img = synth.images(353, 1).to(DEV)
    ex.preprocess_img = lambda p: img
    ex.forward_greedy("synthetic.jpg")
    _, seqs = model.greedy_search(img, synth.word_map(V), max_cap_length=20)
    words = [w for w in seqs[0][1:] if w != 0]
    n = min(len(words), ex.caption_length)
    assert n > 0 and ex.beam_caption_encode[1:1 + n] == words[:n]
    d_img, _ = ex.explain_caption_wordt(0)
    cam = ex.grad_cam(ex.image_features, d_img)
    assert cam.shape == (196,)
    assert_close(cam, O.grad_cam(_pix(ex.image_features.cpu()), _pix(d_img.cpu())), rtol=1e-3, atol=1e-5, what="grad_cam")
    assert_close(ex.explain_cnn(d_img)[0], cam, rtol=0, atol=0, what="explain_cnn of the CAM class")
