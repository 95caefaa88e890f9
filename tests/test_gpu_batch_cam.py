"""GPU: Grad-CAM and Guided Grad-CAM through the batched pipeline (lrpx.pipeline.BatchExplainer).

* the Guided Grad-CAM factor applied in the first layer's epilogue of the guided chain (lrpx_cam_expand_rows_f32 +
  lrpx_tc_conv_args.cam_rows / cam_kw) equals lrpx_cam_expand_mul_f32 of the plain chain's output bit for bit, in every
  delivery format;
* BatchExplainer with the six CAM classes = their per-image explain_cnn / explain_caption_wordt, eager and graph-replayed,
  with ragged captions and through explain_images;
* Grad-CAM on a Bottleneck-ResNet encoder in precision 'mixed' / 'bf16' (tensor-core forward, no chain);
* argument errors and weight updates under captured graphs."""
import argparse

import pytest
import torch
from scipy.stats import spearmanr

import synth
from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
V, H, E, T = 60, 64, 64, 4          # E == H: the adaptive-attention explainer needs it


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _args(tmp_path, encoder="vgg16", E=E, H=H):
    return argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder=encoder, height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")


def _rel_l2(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).norm() / b.norm())


def _mean3(x):
    """the epilogue's channel mean ((c0 + c1) + c2) / 3 with a true division (torch divides by a scalar through its
    reciprocal)"""
    s = (x[:, 0] + x[:, 1]) + x[:, 2]
    return torch.div(s, torch.full_like(s, 3.0))


def _rank_corr(a, b):
    """Spearman with average ranks: Grad-CAM maps hold many exact zeros (the ReLU), which must tie"""
    return float(spearmanr(a.detach().cpu().double().flatten().numpy(), b.detach().cpu().double().flatten().numpy())[0])


# ------------------------------------------------------------------------------------------------ kernel identity
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_fused_factor_equals_cam_expand_mul(precision):
    from lrpx import ops, tc
    from models._gradient import expand_operator
    cfg = [64, 64, "M", 128, "M", 128]
    sd = synth.vgg_state(501, cfg)
    ws = [sd[k].to(DEV) for k in sd if k.endswith("weight")]
    bs = [sd[k].to(DEV) for k in sd if k.endswith("bias")]
    eng = tc.TcVggEngine(ws, bs, cfg, DEV, precision=precision, rule="guided")
    x = synth.images(502, 2, 48).to(DEV)
    st = eng.forward(x)
    fh, fw = st.feat_hw
    Q = 5
    g = torch.Generator().manual_seed(503)
    r_feat = torch.randn(Q, fh * fw, st.feat_c, generator=g).to(DEV)
    rows = torch.tensor([0, 1, 1, 0, 1], dtype=torch.int32, device=DEV)
    cam = torch.rand(Q, fh, fw, generator=g).to(DEV)
    cam[:, 0, :2] = 0                                        # Grad-CAM maps hold exact zeros
    up = 48 // fh
    Kh = torch.tensor(expand_operator(fh, up), dtype=torch.float32, device=DEV)
    Kw = torch.tensor(expand_operator(fw, up), dtype=torch.float32, device=DEV)
    rows_T = ops.cam_expand_rows(cam, Kh)
    assert rows_T.shape == (Q, 48, fw)
    assert_close(rows_T, torch.einsum("yi,qij->qyj", Kh.double(), cam.double()), rtol=1e-6, atol=1e-7, what="T")
    # chunk=2: the factor's rows follow the chain's chunks
    plain = eng.relevance(st, r_feat, rows, chunk=2)
    want = ops.cam_expand_mul(plain, cam, Kh, Kw)
    fused = eng.relevance(st, r_feat, rows, chunk=2, cam=(rows_T, Kw))
    assert torch.equal(fused, want), float((fused - want).abs().max())
    mean = eng.relevance(st, r_feat, rows, chunk=2, deliver="channel_mean", cam=(rows_T, Kw))
    assert torch.equal(mean, _mean3(want)), float((mean - _mean3(want)).abs().max())
    half = eng.relevance(st, r_feat, rows, chunk=2, deliver="fp16", cam=(rows_T, Kw))
    assert torch.equal(half, want.half())
    # without the factor the chain's output is the plain one
    assert torch.equal(eng.relevance(st, r_feat, rows, chunk=2), plain)


# ------------------------------------------------------------------------------------------------ batch = per image
def _module(family):
    from models import gridTDmodel, aoamodel, adaptiveattention
    return {"gridtd": gridTDmodel, "aoa": aoamodel, "adaptive": adaptiveattention}[family]


def _model(family, seed):
    M = _module(family)
    if family == "gridtd":
        model, sd = M.GridTDModel(E, H, V, "vgg16"), synth.gridtd_decoder_state(seed, V, H, E)
    elif family == "aoa":
        model, sd = M.AOAModel(E, H, 8, V, "vgg16"), synth.aoa_decoder_state(seed, V, H, E)
    else:
        model, sd = M.AdaptiveAttentionCaptioningModel(E, H, V, "vgg16"), synth.adaptive_decoder_state(seed, V, H, E)
    model.load_state_dict(sd, strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(seed + 1))
    return model.to(DEV).eval()


CAM_CLASSES = [("gridtd", "ExplainGridTDGradCam"), ("gridtd", "ExplainGridTDGuidedGradCam"),
               ("aoa", "ExplainAOAGradCam"), ("aoa", "ExplainAOAGuidedGradCam"),
               ("adaptive", "ExplainAdaptiveGradCam"), ("adaptive", "ExplainAdaptiveGuidedGradCam")]


def _per_image(ex, imgs, toks, b, t):
    """explain_cnn(explain_caption_wordt(t)[0]) of image b and its word relevances"""
    ex.img = imgs[b:b + 1]
    ex.beam_caption_encode = toks[b].tolist()
    ex._set_state(ex.img, ex.beam_caption_encode)
    d_img, rw = ex._explain_word(t, 0)
    return ex.explain_cnn(d_img), rw


@pytest.mark.parametrize("family,cls", CAM_CLASSES)
def test_batch_explainer_with_cam_explainers(tmp_path, family, cls):
    from lrpx.pipeline import BatchExplainer
    model = _model(family, 521)
    ex = getattr(_module(family), cls)(_args(tmp_path), synth.word_map(V), model=model, precision="fp32")
    imgs = synth.images(522, 2).to(DEV)
    toks = torch.tensor([synth.tokens(523, T, V), synth.tokens(524, T, V)], device=DEV)
    # tc_gemm=False: the decoder GEMMs on fp32 CUDA cores, as the one-word path of precision 'fp32' runs them
    heat, r_words = BatchExplainer(ex, chunk=4, tc_gemm=False).explain(imgs, toks)
    heat, r_words = heat.clone(), r_words.clone()
    shape = (2 * T, 196) if ex.CAM == "cam" else (2 * T, 3, 224, 224)
    assert heat.shape == shape and r_words.shape == (2 * T, T)
    heat_g, words_g = BatchExplainer(ex, chunk=4, use_graph=True, tc_gemm=False).explain(imgs, toks)
    assert torch.equal(heat_g, heat) and torch.equal(words_g, r_words), "graph replay"
    for b in range(2):
        for t in (0, T - 1):
            one, rw = _per_image(ex, imgs, toks, b, t)
            q = b * T + t
            # the explainer forward's library GEMMs pick another algorithm for 2 rows than for 1: ~1e-5 of the maximum
            assert_close(heat[q:q + 1], one, rtol=1e-3, atol=1e-4 * float(one.abs().max()), what=f"image {b} word {t}")
            assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=1e-5, what=f"words image {b} word {t}")
    # ragged captions: the valid (image, word) pairs only, in the same image-major order
    wpi = (T, 2)
    heat_r, words_r = BatchExplainer(ex, chunk=4, tc_gemm=False).explain(imgs, toks, words_per_image=wpi)
    keep = [b * T + t for b in range(2) for t in range(wpi[b])]
    assert heat_r.shape[0] == len(keep)
    assert_close(heat_r, heat[keep], rtol=1e-3, atol=1e-4 * float(heat.abs().max()), what="ragged")
    assert_close(words_r, r_words[keep], rtol=1e-3, atol=1e-5, what="ragged words")
    # explain_images: the maps of its own captions, as explain() computes them
    be = BatchExplainer(ex, chunk=4, tc_gemm=False)
    res = be.explain_images(imgs, beam_size=2, max_cap_length=3)
    assert res.heat.shape == (sum(res.words_per_image),) + shape[1:]
    h2, w2 = BatchExplainer(ex, chunk=4, tc_gemm=False).explain(imgs, res.tokens, words_per_image=res.words_per_image)
    assert torch.equal(res.heat, h2) and torch.equal(res.r_words, w2)


@pytest.mark.parametrize("cls", ["ExplainGridTDGradCam", "ExplainGridTDGuidedGradCam"])
def test_cam_delivery_formats_and_host_copy(tmp_path, cls):
    """precision 'bf16': Guided Grad-CAM's 'channel_mean' / 'fp16' are the formats of its 'full' maps; host delivery of
    either method equals the device result"""
    from lrpx.pipeline import BatchExplainer
    from models import gridTDmodel as G
    ex = getattr(G, cls)(_args(tmp_path), synth.word_map(V), model=_model("gridtd", 531), precision="bf16")
    imgs = synth.images(532, 2).to(DEV)
    toks = torch.tensor([synth.tokens(533, T, V), synth.tokens(534, T, V)], device=DEV)
    full, words = BatchExplainer(ex, chunk=3).explain(imgs, toks)
    full, words = full.clone(), words.clone()
    host = (torch.empty(full.shape, pin_memory=True), torch.empty(words.shape, pin_memory=True))
    for graph in (False, True):
        BatchExplainer(ex, chunk=3, use_graph=graph).explain(imgs, toks, host_out=host)
        torch.cuda.synchronize()
        assert torch.equal(host[0], full.cpu()) and torch.equal(host[1], words.cpu())
    if ex.CAM == "guided":
        mean = BatchExplainer(ex, chunk=3, deliver="channel_mean").explain(imgs, toks)[0]
        assert torch.equal(mean, _mean3(full)), float((mean - _mean3(full)).abs().max())
        half = BatchExplainer(ex, chunk=3, deliver="fp16", use_graph=True).explain(imgs, toks)[0]
        assert torch.equal(half, full.half())


# ------------------------------------------------------------------------------------------------ ResNet encoders
def _gridtd_resnet101():
    from models import gridTDmodel as G
    torch.manual_seed(23)
    Er = 32
    model = G.GridTDModel(Er, H, V, "resnet101", n_pixel=49)
    model.load_state_dict(synth.gridtd_decoder_state(331, V, H, Er, C=2048, n_pixel=49), strict=False)
    return model.to(DEV).eval()


def test_grad_cam_on_resnet_mixed_and_bf16(tmp_path):
    from lrpx.pipeline import BatchExplainer
    from models import gridTDmodel as G
    model = _gridtd_resnet101()
    args = _args(tmp_path, "resnet101", E=32)
    imgs = synth.images(541, 2).to(DEV)
    toks = torch.tensor([synth.tokens(542 + b, 3, V) for b in range(2)], device=DEV)
    ref = G.ExplainGridTDGradCam(args, synth.word_map(V), model=model, precision="simt")
    want = {(b, t): _per_image(ref, imgs, toks, b, t) for b in range(2) for t in range(3)}
    # 'mixed': fp32-accurate features, the maps agree to 1e-4; 'bf16': the bf16 forward's feature error (7e-3) moves the
    # 49-pixel maps by a few percent and swaps near-equal pixels (measured on a B200: rel L2 <= 2.7e-2, Spearman down to 0.96)
    bars = {"mixed": (0.99, 1e-3), "bf16": (0.9, 0.1)}
    for prec in ("mixed", "bf16"):
        ex = G.ExplainGridTDGradCam(args, synth.word_map(V), model=model, precision=prec)
        assert ex.uses_tc and ex.is_resnet
        rhos, l2s = [], []
        for (b, t), (m_ref, w_ref) in want.items():
            m, w = _per_image(ex, imgs, toks, b, t)
            rhos.append(_rank_corr(m, m_ref))
            l2s.append(_rel_l2(m, m_ref))
            print(f"ResNet101 Grad-CAM {prec} vs simt, image {b} word {t}: Spearman {rhos[-1]:.5f}, rel L2 {l2s[-1]:.3e}")
        assert min(rhos) >= bars[prec][0] and max(l2s) <= bars[prec][1], (prec, rhos, l2s)
        heat, r_words = BatchExplainer(ex, chunk=4).explain(imgs, toks)
        heat, r_words = heat.clone(), r_words.clone()
        assert heat.shape == (6, 49)
        heat_g, words_g = BatchExplainer(ex, chunk=4, use_graph=True).explain(imgs, toks)
        assert torch.equal(heat_g, heat) and torch.equal(words_g, r_words), "graph replay"
        for (b, t) in want:
            one, rw = _per_image(ex, imgs, toks, b, t)
            q = b * 3 + t
            assert_close(heat[q:q + 1], one, rtol=1e-3, atol=1e-4 * float(one.abs().max()), what=f"{prec} {b} {t}")
            assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=1e-5, what=f"{prec} words {b} {t}")
    # the gradient chain of a ResNet does not exist on the tensor cores: the other gradient classes keep refusing
    for cls in ("ExplainGridTDGradient", "ExplainiGridTDGuidedGradient", "ExplainGridTDGuidedGradCam"):
        with pytest.raises(NotImplementedError):
            getattr(G, cls)(args, synth.word_map(V), model=model, precision="mixed")


# ------------------------------------------------------------------------------------------------ errors
def test_cam_argument_errors(tmp_path):
    from lrpx import _lib, tc
    from lrpx.pipeline import BatchExplainer
    from models import gridTDmodel as G
    ex = G.ExplainGridTDGradCam(_args(tmp_path), synth.word_map(V), model=_model("gridtd", 551), precision="bf16")
    for deliver in ("channel_mean", "fp16"):
        with pytest.raises(ValueError):
            BatchExplainer(ex, deliver=deliver)
    cfg = [64, "M", 64]
    sd = synth.vgg_state(552, cfg)
    ws = [sd[k].to(DEV) for k in sd if k.endswith("weight")]
    bs = [sd[k].to(DEV) for k in sd if k.endswith("bias")]
    x = synth.images(553, 1, 16).to(DEV)
    for rule in ("gradient", "guided"):
        eng = tc.TcVggEngine(ws, bs, cfg, DEV, precision="bf16", rule=rule)
        st = eng.forward(x)
        r = torch.randn(1, 64, 64, device=DEV)
        Kw = torch.ones(16, 8, device=DEV)
        good = torch.ones(1, 16, 8, device=DEV)
        if rule == "gradient":
            with pytest.raises(_lib.LrpxError):
                eng.relevance(st, r, cam=(good, Kw))
        else:
            with pytest.raises(_lib.LrpxError):
                eng.relevance(st, r, cam=(torch.ones(1, 16, 4, device=DEV), Kw))      # T and Kw disagree on w
            assert eng.relevance(st, r, cam=(good, Kw)).shape == (1, 3, 16, 16)


# ------------------------------------------------------------------------------------------------ weight updates
def test_graph_replay_after_weight_updates_equals_fresh(tmp_path):
    """A graph-replaying BatchExplainer picks up in-place updates: an encoder conv bias (Guided Grad-CAM, VGG) and a
    BatchNorm buffer (Grad-CAM, ResNet101 in 'mixed')."""
    from lrpx.pipeline import BatchExplainer
    from models import gridTDmodel as G
    cases = []
    model = _model("gridtd", 561)
    ex = G.ExplainGridTDGuidedGradCam(_args(tmp_path), synth.word_map(V), model=model, precision="bf16")
    cases.append((ex, lambda: model.img_encoder.encoder[2].bias.add_(0.05), T))
    rmodel = _gridtd_resnet101()
    rex = G.ExplainGridTDGradCam(_args(tmp_path, "resnet101", E=32), synth.word_map(V), model=rmodel, precision="mixed")
    cases.append((rex, lambda: rmodel.img_encoder.encoder.layer1[0].bn2.running_var.mul_(1.7), 3))
    for ex, update, n in cases:
        imgs = synth.images(562, 2).to(DEV)
        toks = torch.tensor([synth.tokens(563 + b, n, V) for b in range(2)], device=DEV)
        be = BatchExplainer(ex, chunk=4, use_graph=True)
        before = [t.clone() for t in be.explain(imgs, toks)]
        with torch.no_grad():
            update()
        after = [t.clone() for t in be.explain(imgs, toks)]
        fresh = BatchExplainer(ex, chunk=4, use_graph=True).explain(imgs, toks)
        assert not torch.equal(before[0], fresh[0]), "the update did not change the explanation"
        assert torch.equal(after[0], fresh[0]) and torch.equal(after[1], fresh[1])
