"""Explanations after an in-place weight update (``load_state_dict``, ``p.add_()`` under ``no_grad``, what an optimizer
step does) equal those of an explainer built fresh on the updated model, bit for bit.  The explainers, BatchExplainer
and the decoders' persistent workspaces keep prepared copies of the weights (concatenated gate rows, the encoder
engine's converted conv weights, split bf16 copies for the tensor-core GEMMs): each must notice the update."""
import argparse

import pytest
import torch

import helpers
import lrp_oracle as O
import synth

pytestmark = pytest.mark.gpu
DEV = "cuda"
V, H, E = 60, 64, 32


def _build(family, gradient, tmp_path, precision):
    """A small decoder on VGG16 at 224 x 224 and its explainer."""
    from models import adaptiveattention as AA
    from models import aoamodel as A
    from models import gridTDmodel as G
    e = H if family == "adaptive" else E                 # the adaptive explainer needs embed_dim == hidden_dim
    args = argparse.Namespace(embed_dim=e, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")
    if family == "gridtd":
        model = G.GridTDModel(e, H, V, "vgg16")
        cls = G.ExplainGridTDGradient if gradient else G.ExplainGridTDAttention
    elif family == "aoa":
        model = A.AOAModel(e, H, 8, V, "vgg16")
        cls = A.ExplainAOAGradient if gradient else A.ExplainAOAAttention
    else:
        model = AA.AdaptiveAttentionCaptioningModel(e, H, V, "vgg16")
        cls = AA.ExplainAdaptiveGradient if gradient else AA.ExplainAdaptiveAttention
    model.load_state_dict(_decoder_state(family, 91, e), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(92))
    model.to(DEV).eval()
    make = lambda: cls(args, synth.word_map(V), model=model, precision=precision)
    return model, make, e


def _decoder_state(family, seed, e):
    if family == "gridtd":
        return synth.gridtd_decoder_state(seed, V, H, e)
    if family == "aoa":
        return synth.aoa_decoder_state(seed, V, H, e)
    return synth.adaptive_decoder_state(seed, V, H, e)


def _update(model, family, e, what):
    if what == "decoder":
        model.load_state_dict(_decoder_state(family, 93, e), strict=False)
        return
    g = torch.Generator().manual_seed(94)
    with torch.no_grad():
        for p in model.img_encoder.encoder.parameters():
            p.add_(torch.randn(p.shape, generator=g).to(p.device) * 0.1 * float(p.std() if p.numel() > 1 else 1e-2))


def _explain(ex, img, tk, family):
    ex.preprocess_img = lambda path: img
    ex.model.beam_search = lambda *a, **k: (["w1 w2 w3"], tk[1:])
    ex.ACCUMULATE_LIKE_REFERENCE = False
    out = ex.explain_caption("synthetic.jpg", 2) if family == "aoa" else ex.explain_caption("synthetic.jpg")
    heat, words = out
    return torch.cat(heat), [w.clone() for w in words]


@pytest.mark.parametrize("update", ["decoder", "encoder"])
@pytest.mark.parametrize("precision", ["fp32", "simt"])
@pytest.mark.parametrize("gradient", [False, True], ids=["lrp", "gradient"])
@pytest.mark.parametrize("family", ["gridtd", "aoa", "adaptive"])
def test_explainer_after_weight_update_equals_fresh_explainer(tmp_path, family, gradient, precision, update):
    model, make, e = _build(family, gradient, tmp_path, precision)
    img = synth.images(95, 1).to(DEV)
    tk = synth.tokens(96, 3, V)
    ex = make()
    before = _explain(ex, img, tk, family)                # fills every cache of the explainer
    _update(model, family, e, update)
    after = _explain(ex, img, tk, family)
    fresh = _explain(make(), img, tk, family)
    assert not torch.equal(before[0], fresh[0]), "the update did not change the explanation"
    assert torch.equal(after[0], fresh[0]), f"heat-maps: max diff {float((after[0] - fresh[0]).abs().max()):.3e}"
    for a, f in zip(after[1], fresh[1]):
        assert torch.equal(a, f)


@pytest.mark.parametrize("update", ["decoder", "encoder"])
@pytest.mark.parametrize("gradient", [False, True], ids=["lrp", "gradient"])
def test_batch_explainer_after_weight_update_equals_fresh(tmp_path, gradient, update):
    """Eager, and replaying a graph captured before the update: equal to a BatchExplainer built after it."""
    from lrpx.pipeline import BatchExplainer
    model, make, e = _build("gridtd", gradient, tmp_path, "bf16" if not gradient else "fp32")
    B, T = 2, 3
    imgs = synth.images(97, B).to(DEV)
    toks = torch.stack([torch.tensor(synth.tokens(98 + b, T, V)) for b in range(B)]).to(DEV)
    ex = make()
    eager, graph = BatchExplainer(ex, chunk=4), BatchExplainer(ex, chunk=4, use_graph=True)
    before = eager.explain(imgs, toks)[0].clone()
    graph.explain(imgs, toks)                              # captures
    _update(model, "gridtd", e, update)
    he, we = eager.explain(imgs, toks)
    he, we = he.clone(), we.clone()
    hg, wg = graph.explain(imgs, toks)
    hf, wf = BatchExplainer(make(), chunk=4).explain(imgs, toks)
    assert not torch.equal(before, hf), "the update did not change the explanation"
    assert torch.equal(he, hf) and torch.equal(we, wf), "eager"
    assert torch.equal(hg, hf) and torch.equal(wg, wf), "graph replay"


@pytest.mark.parametrize("family", ["gridtd", "aoa", "adaptive"])
def test_decoder_workspace_cache_with_other_weights(family):
    """ops.*_decoder_lrp(..., ws_cache=cache) called with a second weight dict of the same shapes equals the uncached
    call: the prepared weight copies in a cached workspace belong to the weights they were made from."""
    from lrpx import decoder as D
    from lrpx import ops
    h, e, c, P = 64, 64, 256, 16
    f = torch.randn(c, 4, 4, generator=torch.Generator().manual_seed(99)).clamp(min=0)
    tk = synth.tokens(100, 4, V)
    if family == "gridtd":
        ps = [synth.gridtd_decoder_state(s, V, h, e, C=c, n_pixel=P) for s in (101, 102)]
        ks = helpers.gridtd_kernel_state([O.gridtd_explainer_forward(ps[0], f, tk)], DEV)
        Ws = [helpers.to_dev(D.gridtd_weights(p), DEV) for p in ps]
        call = lambda W, **kw: ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, tc_gemm=True, **kw)
    elif family == "aoa":
        ps = [synth.aoa_decoder_state(s, V, h, e, C=c) for s in (101, 102)]
        ks = helpers.aoa_kernel_state([O.aoa_explainer_forward(ps[0], f, tk, 8)], DEV)
        Ws = [helpers.to_dev(D.aoa_weights(p), DEV) for p in ps]
        call = lambda W, **kw: ops.aoa_decoder_lrp(ks, W, 8, req_img, req_t, req_word, req_t * 2, tc_gemm=True, **kw)
    else:
        ps = [synth.adaptive_decoder_state(s, V, h, e, C=c, n_pixel=P) for s in (101, 102)]
        ks = helpers.adaptive_kernel_state([O.adaptive_explainer_forward(ps[0], f, tk)], DEV)
        Ws = [helpers.to_dev(D.adaptive_weights(p), DEV) for p in ps]
        call = lambda W, **kw: ops.adaptive_decoder_lrp(ks, W, req_img, req_t, req_word, tc_gemm=True, **kw)
    req_t = torch.arange(4, dtype=torch.int32, device=DEV)
    req_img = torch.zeros_like(req_t)
    req_word = torch.tensor(tk[1:], dtype=torch.int32, device=DEV)
    cache = {}
    ref = [call(W) for W in Ws]
    first = call(Ws[0], ws_cache=cache)
    second = call(Ws[1], ws_cache=cache)
    again = call(Ws[0], ws_cache=cache)
    assert not torch.equal(ref[0][0], ref[1][0])
    for got, want in ((first, ref[0]), (second, ref[1]), (again, ref[0])):
        assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    # the weights changed in place: the cached copies are stale
    with torch.no_grad():
        Ws[0]["W_g" if family != "gridtd" else "W_g1"].mul_(1.5)
    assert torch.equal(call(Ws[0], ws_cache=cache)[0], call(Ws[0])[0])
