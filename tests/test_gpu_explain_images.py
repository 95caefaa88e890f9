"""BatchExplainer.explain_images: a batch of images captioned by the explainer's device beam search and explained on
the features of the same encoder pass — equal to the two-step API (search, then explain) bit for bit, to the per-image
API's captions and explanations, with one encoder forward per call."""
import argparse

import pytest
import torch

import synth
from conftest import assert_close

pytestmark = pytest.mark.gpu
DEV = "cuda"
V, H, E = 80, 64, 64          # E == H: the adaptive-attention explainer needs it


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _args(tmp_path, encoder="vgg16", E=E, H=H):
    return argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder=encoder, height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")


def _module(family):
    from models import gridTDmodel, aoamodel, adaptiveattention
    return {"gridtd": gridTDmodel, "aoa": aoamodel, "adaptive": adaptiveattention}[family]


def _model(family, seed, end_bias=0.0):
    """A VGG16 model whose random init keeps real words ahead of the special tokens (captions run to the length cap),
    ``end_bias`` added to the <end> logit."""
    M, wm = _module(family), synth.word_map(V)
    if family == "gridtd":
        model, sd = M.GridTDModel(E, H, V, "vgg16"), synth.gridtd_decoder_state(seed, V, H, E)
    elif family == "aoa":
        model, sd = M.AOAModel(E, H, 8, V, "vgg16"), synth.aoa_decoder_state(seed, V, H, E)
    else:
        model, sd = M.AdaptiveAttentionCaptioningModel(E, H, V, "vgg16"), synth.adaptive_decoder_state(seed, V, H, E)
    model.load_state_dict(sd, strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(seed + 1))
    model.to(DEV).eval()
    with torch.no_grad():
        for tok in ('<end>', '<unk>', '<pad>', '<start>'):
            model.fc.bias[wm[tok]] -= 2.0
        model.fc.bias[wm['<end>']] += end_bias
    return model


def _explainer(family, cls, precision, tmp_path, seed=601, end_bias=0.0, model=None):
    model = _model(family, seed, end_bias) if model is None else model
    return getattr(_module(family), cls)(_args(tmp_path), synth.word_map(V), model=model, precision=precision)


def _check_layout(res, B, start):
    """tokens hold <start>, the caption and 0-padding; requests are the caption words in image-major order"""
    T = res.tokens.shape[1] - 1
    assert res.tokens.shape == (B, T + 1) and T == max(res.words_per_image)
    assert list(res.words_per_image) == [len(c) for c in res.captions]
    for b, c in enumerate(res.captions):
        assert res.tokens[b].tolist() == [start] + c + [0] * (T - len(c))
    want = [(b, t) for b in range(B) for t in range(res.words_per_image[b])]
    assert list(zip(res.req_img.tolist(), res.req_t.tolist())) == want
    assert res.r_words.shape == (len(want), T) and res.heat.shape[0] == len(want)
    assert res.pred.shape[:2] == (B, T)


def _check_two_step(ex, imgs, res, **kw):
    """heat / r_words bit-equal to explain() on the found captions (fresh BatchExplainer), pred to the explainer forward"""
    from lrpx.pipeline import BatchExplainer
    heat, r_words = BatchExplainer(ex, chunk=8, **kw).explain(imgs, res.tokens, words_per_image=res.words_per_image)
    assert torch.equal(res.heat, heat) and torch.equal(res.r_words, r_words)
    eng = ex.engine()
    feat = eng.features(eng.forward(imgs), "pixel")
    assert torch.equal(res.pred, ex.explainer_forward(feat, res.tokens)["pred"])


CASES = [("gridtd", "ExplainGridTDAttention", "bf16"), ("aoa", "ExplainAOAAttention", "bf16"),
         ("adaptive", "ExplainAdaptiveAttention", "bf16"), ("gridtd", "ExplainGridTDGradient", "bf16"),
         ("aoa", "ExplainAOAGuidedGradient", "bf16"), ("gridtd", "ExplainGridTDAttention", "fp32")]


@pytest.mark.parametrize("family,cls,precision", CASES)
def test_equals_search_then_explain(tmp_path, family, cls, precision):
    from lrpx.pipeline import BatchExplainer
    ex = _explainer(family, cls, precision, tmp_path)
    imgs = synth.images(602, 3).to(DEV)
    kw = dict(head_idx=1) if family == "aoa" else {}
    res = BatchExplainer(ex, chunk=8, **kw).explain_images(imgs, beam_size=2, max_cap_length=6)
    _check_layout(res, 3, ex.word_map['<start>'])
    assert sum(res.words_per_image) > 0
    _check_two_step(ex, imgs, res, **kw)
    # the captions are the searcher's on the features of that pass
    eng = ex.engine()
    with torch.no_grad():
        proj, glob = ex._search_inputs(eng.features(eng.forward(imgs), "pixel"))
    assert res.captions == ex._searcher().search(proj, glob, ex.word_map, beam_size=2, max_cap_length=6)


@pytest.mark.parametrize("family", ["gridtd", "aoa", "adaptive"])
def test_captions_equal_the_per_image_search_with_its_defaults(tmp_path, family):
    """Default beam size / length = the ones get_hidden_parameters passes; each caption = _find_caption on the image
    alone."""
    from lrpx.pipeline import BatchExplainer
    cls = {"gridtd": "ExplainGridTDAttention", "aoa": "ExplainAOAAttention", "adaptive": "ExplainAdaptiveAttention"}
    ex = _explainer(family, cls[family], "bf16", tmp_path, seed=611, end_bias=1.5)
    imgs = synth.images(612, 3).to(DEV)
    used = {}
    searcher = ex._searcher()
    search = searcher.search

    def spy(*a, beam_size, max_cap_length, **k):
        used.setdefault("search", []).append((beam_size, max_cap_length))
        return search(*a, beam_size=beam_size, max_cap_length=max_cap_length, **k)
    searcher.search = spy
    res = BatchExplainer(ex, chunk=8).explain_images(imgs)
    find = ex._find_caption

    def find_spy(path, beam_size, max_cap_length):
        used["find"] = (beam_size, max_cap_length)
        return find(path, beam_size, max_cap_length)
    ex._find_caption = find_spy
    ex.preprocess_img = lambda p: imgs[:1]
    ex.get_hidden_parameters("synthetic.jpg")
    assert used["search"][0] == used["find"] == ex.CAPTION_SEARCH
    for b in range(3):
        ex.img = imgs[b:b + 1]
        find("synthetic.jpg", *ex.CAPTION_SEARCH)
        assert res.captions[b] == ex.beam_caption_encode[1:], b
    print(f"{family}: caption lengths {res.words_per_image}")


def test_equals_explain_caption(tmp_path):
    """Two words of one image against the per-image explain_caption (per-word heat-maps), the tolerances of
    test_gpu_models.py::test_batch_pipeline_graph_equals_eager_and_single_image_api."""
    from lrpx.pipeline import BatchExplainer
    ex = _explainer("gridtd", "ExplainGridTDAttention", "bf16", tmp_path, seed=621)
    ex.ACCUMULATE_LIKE_REFERENCE = False
    imgs = synth.images(622, 2).to(DEV)
    res = BatchExplainer(ex, chunk=8).explain_images(imgs)
    b = 1
    ex.preprocess_img = lambda p: imgs[b:b + 1]
    hs, ws = ex.explain_caption("synthetic.jpg")
    T = res.words_per_image[b]
    assert ex.beam_caption_encode[1:] == res.captions[b] and len(hs) == T > 1
    q0 = res.words_per_image[0]
    for t in (0, T - 1):
        q = q0 + t
        assert (int(res.req_img[q]), int(res.req_t[q])) == (b, t)
        assert_close(hs[t][0], res.heat[q], rtol=1e-3, atol=1e-6 + 1e-3 * float(res.heat[q].abs().max()),
                     what=f"image {b} word {t}")
        assert_close(ws[t], res.r_words[q, :t + 1], rtol=1e-3, atol=1e-4, what=f"words {b},{t}")


def test_one_encoder_pass(tmp_path):
    """The model's own (library) _encode never runs, and the call launches as many lrpx_tc_conv as explain(), which
    runs one encoder forward and the chain."""
    from lrpx import _lib
    from lrpx.pipeline import BatchExplainer
    ex = _explainer("gridtd", "ExplainGridTDAttention", "bf16", tmp_path, seed=631)
    imgs = synth.images(632, 3).to(DEV)

    def no_encode(*a, **k):
        raise AssertionError("the model's library encoder ran")
    ex.model._encode = no_encode
    pipe = BatchExplainer(ex, chunk=8)
    pipe.explain_images(imgs, max_cap_length=5)                      # warm-up: engine and search plans built
    n = lambda: _lib.CALLS.get("lrpx_tc_conv", 0)
    c0 = n()
    res = pipe.explain_images(imgs, max_cap_length=5)
    c_images = n() - c0
    c0 = n()
    pipe.explain(imgs, res.tokens, words_per_image=res.words_per_image)
    c_explain = n() - c0
    c0 = n()
    ex.engine().forward(imgs)
    c_forward = n() - c0
    print(f"lrpx_tc_conv launches: explain_images {c_images}, explain {c_explain}, one forward {c_forward}")
    assert c_forward > 0 and c_images == c_explain


def _gridtd_resnet101(V, H, E):
    from models import gridTDmodel as G
    torch.manual_seed(23)
    model = G.GridTDModel(E, H, V, "resnet101", n_pixel=49)
    model.load_state_dict(synth.gridtd_decoder_state(331, V, H, E, C=2048, n_pixel=49), strict=False)
    return model.to(DEV).eval()


def test_resnet101_mixed(tmp_path):
    from models import gridTDmodel as G
    from lrpx.pipeline import BatchExplainer
    Vr, Hr, Er = 60, 64, 32
    model, wm = _gridtd_resnet101(Vr, Hr, Er), synth.word_map(Vr)
    with torch.no_grad():
        for tok in ('<end>', '<unk>', '<pad>', '<start>'):
            model.fc.bias[wm[tok]] -= 2.0
    ex = G.ExplainGridTDAttention(_args(tmp_path, "resnet101", Er, Hr), wm, model=model, precision="mixed")
    imgs = synth.images(641, 3).to(DEV)
    res = BatchExplainer(ex, chunk=8).explain_images(imgs, max_cap_length=6)
    assert sum(res.words_per_image) > 0
    _check_layout(res, 3, wm['<start>'])
    _check_two_step(ex, imgs, res)


def test_all_captions_empty(tmp_path):
    from lrpx.pipeline import BatchExplainer
    ex = _explainer("gridtd", "ExplainGridTDAttention", "bf16", tmp_path, seed=651, end_bias=60.0)
    imgs = synth.images(652, 3).to(DEV)
    for deliver in ("full", "channel_mean"):
        pipe = BatchExplainer(ex, chunk=8, deliver=deliver)
        res = pipe.explain_images(imgs)
        assert res.captions == [[], [], []] and res.words_per_image == (0, 0, 0)
        assert res.tokens.tolist() == [[synth.word_map(V)['<start>']]] * 3
        assert res.req_img.numel() == 0 and res.req_t.numel() == 0 and res.pred.shape == (3, 0, V)
        heat, r_words = pipe.explain(imgs, res.tokens, words_per_image=res.words_per_image)
        assert res.heat.shape == heat.shape and res.heat.dtype == heat.dtype
        assert res.r_words.shape == r_words.shape == (0, 0)


def test_ragged_captions(tmp_path):
    """Biases on <end> that make some captions end before the cap: requests in image-major order of words_per_image,
    results equal to explain() on the same requests."""
    from lrpx.pipeline import BatchExplainer
    model = _model("gridtd", 661)
    ex = _explainer("gridtd", "ExplainGridTDAttention", "bf16", tmp_path, model=model)
    end = synth.word_map(V)['<end>']
    base = model.fc.bias[end].item()
    imgs = synth.images(662, 4).to(DEV)
    imgs[1] *= 3.0                     # features further from the others': a different search outcome
    imgs[3] = imgs[3].abs()
    n_ragged = 0
    # the captions of this model go from never ending to ending at once between <end> biases of 2.0 and 2.5
    for end_bias in [2.0 + 0.05 * i for i in range(11)]:
        with torch.no_grad():
            model.fc.bias[end] = base + end_bias
        res = BatchExplainer(ex, chunk=8).explain_images(imgs, beam_size=3, max_cap_length=8)
        n = res.words_per_image
        print(f"<end> bias {end_bias}: caption lengths {n}")
        if len(set(n)) < 2 or max(n) == 0:
            continue
        n_ragged += 1
        _check_layout(res, 4, ex.word_map['<start>'])
        _check_two_step(ex, imgs, res)
    assert n_ragged > 0, "no ragged batch: the padding and request order were not exercised"


def test_host_out(tmp_path):
    from lrpx.pipeline import BatchExplainer
    ex = _explainer("gridtd", "ExplainGridTDAttention", "bf16", tmp_path, seed=671)
    imgs = synth.images(672, 3).to(DEV)
    L = 8
    hh = torch.full((3 * L, 3, 224, 224), float("nan")).pin_memory()
    wh = torch.full((3 * L, L + 2), float("nan")).pin_memory()         # wider than any caption
    for src in (imgs, imgs.cpu().pin_memory()):
        res = BatchExplainer(ex, chunk=4).explain_images(src, max_cap_length=L, host_out=(hh, wh))
        torch.cuda.synchronize()
        Q, T = res.heat.shape[0], res.r_words.shape[1]
        assert Q > 4                                  # more than one chunk of the copy overlap
        assert torch.equal(hh[:Q], res.heat.cpu()) and torch.equal(wh[:Q, :T], res.r_words.cpu())
    out = torch.empty(3 * L, 3, 224, 224, device=DEV)
    res2 = BatchExplainer(ex, chunk=4).explain_images(imgs, max_cap_length=L, out=out)
    assert res2.heat.data_ptr() == out.data_ptr() and torch.equal(res2.heat, res.heat)
    with pytest.raises(ValueError):
        BatchExplainer(ex, chunk=4).explain_images(imgs, max_cap_length=L, out=out[:1])


def test_feeds_the_image_ablation(tmp_path):
    from lrpx.ablation import AblationExperiments
    from lrpx.pipeline import BatchExplainer
    ex = _explainer("gridtd", "ExplainGridTDAttention", "bf16", tmp_path, seed=681)
    imgs = synth.images(682, 2).to(DEV)
    res = BatchExplainer(ex, chunk=8).explain_images(imgs, max_cap_length=5)
    ab = AblationExperiments(ex, chunk=4)
    got = ab.image_ablation(imgs, res.tokens, res.heat, res.req_img, res.req_t, res.pred)
    heat, _ = BatchExplainer(ex, chunk=8).explain(imgs, res.tokens, words_per_image=res.words_per_image)
    eng = ex.engine()
    pred = ex.explainer_forward(eng.features(eng.forward(imgs), "pixel"), res.tokens)["pred"]
    want = ab.image_ablation(imgs, res.tokens, heat, res.req_img, res.req_t, pred)
    assert torch.equal(got["disappear"], want["disappear"]) and got["captions"] == want["captions"]
    torch.testing.assert_close(got["score_diff"], want["score_diff"], rtol=0, atol=0, equal_nan=True)
