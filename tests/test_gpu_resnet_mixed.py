"""GPU parity: Bottleneck-ResNet encoders in precision 'mixed' (lrpx.tc_resnet.TcResNetMixed): the forward with
error-compensated bf16x3 operands (hi|lo activations, fp32 gains) under the bf16 relevance chain, its stem kernels
(lrpx_tc_im2col7s2_split_x, lrpx_tc_maxpool3s2_x), the routes to it and the batched pipeline on it."""
import argparse
import ctypes as C

import pytest
import torch
import torch.nn.functional as F

import lrp_oracle as O
import synth
from conftest import assert_close, spearman

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(autouse=True)
def _no_tf32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _pf_valid(pf, n, h, w, c):
    """(n, c, h, w) of the valid rows of a PF tensor with c channels per row"""
    return pf.view(n, h + 1, w + 1, c)[:, 1:, 1:, :].permute(0, 3, 1, 2)


def _resnet(layers, seed):
    from models import resnet
    net = resnet.ResNet(resnet.Bottleneck, list(layers))
    net.load_state_dict(synth.resnet_state(seed, tuple(layers)))
    return net.to(DEV).eval()


def _rel_l2(a, b):
    a, b = a.cpu().double(), b.cpu().double()
    return float((a - b).norm() / b.norm())


def _feature_target(feats, g, Q, scale=1e-3):
    """Relevance at the encoder output proportional to the feature (R = a (.) c), as a decoder hands it over (see
    tests/test_gpu_resnet_tc.py::_feature_target)."""
    feats = feats.cpu()
    rimg = torch.arange(Q, dtype=torch.int32) % feats.shape[0]
    return torch.randn((Q,) + tuple(feats.shape[1:]), generator=g) * scale * feats[rimg.long()], rimg


def _pix(t):
    return t.flatten(2).transpose(1, 2).contiguous().to(DEV)


# ------------------------------------------------------------------------------------------------ stem kernels
def test_stem_im2col_split():
    from lrpx import tc, _lib
    lib = _lib.lib()
    g = torch.Generator().manual_seed(31)
    n, H, W = 2, 32, 64
    x = torch.randn(n, 3, H, W, generator=g)
    x[0, :, :5, :7] = 0                                             # exact zero taps
    xd = x.to(DEV)
    h, w = H // 2, W // 2
    rows = tc.pf_rows(n, h, w)
    ref16 = torch.empty(rows, 320, device=DEV, dtype=torch.bfloat16)
    _lib.check(lib.lrpx_tc_im2col7s2_split_bf16(_p(xd), _p(ref16), n, H, W, _stream()), "im2col7s2")
    c0 = torch.full((rows, 320), 7.0, device=DEV, dtype=torch.bfloat16)
    _lib.check(lib.lrpx_tc_im2col7s2_split_x(_p(xd), _p(c0), n, H, W, 0, _stream()), "im2col7s2_x split=0")
    c1 = torch.full((rows, 640), 7.0, device=DEV, dtype=torch.bfloat16)
    _lib.check(lib.lrpx_tc_im2col7s2_split_x(_p(xd), _p(c1), n, H, W, 1, _stream()), "im2col7s2_x split=1")
    torch.cuda.synchronize()
    assert torch.equal(c0, ref16), "split=0 must be the bf16 kernel bit for bit"
    assert torch.equal(c1[:, :320], ref16), "hi must be the bf16 kernel's row bit for bit"
    # fp32 taps: [x+ over (ci, ky, kx) | x- over them | 26 zeros] per output pixel
    cols = F.unfold(x, 7, padding=3, stride=2).transpose(1, 2)                  # (n, h*w, 147)
    taps = torch.cat((cols.clamp(min=0), cols.clamp(max=0), torch.zeros(n, h * w, 26)), 2).reshape(n, h, w, 320)
    v = c1.view(n, h + 1, w + 1, 640).cpu().float()
    assert float(v[:, 0].abs().max()) == 0.0 and float(v[:, :, 0].abs().max()) == 0.0, "padding rows must be zero"
    val = v[:, 1:, 1:, :320] + v[:, 1:, 1:, 320:]
    err = (val - taps).abs()
    assert bool((err <= 2.0 ** -16 * taps.abs()).all()), f"|hi + lo - tap| / |tap| max {float((err / taps.abs().clamp(min=1e-30)).max()):.3e}"


@pytest.mark.parametrize("n,h,w", [(2, 8, 12), (1, 112, 112)])
def test_stem_maxpool_split(n, h, w):
    from lrpx import tc, _lib
    lib = _lib.lib()
    c = 64
    g = torch.Generator().manual_seed(h + w + 1)
    v = torch.randn(n, c, h, w, generator=g).clamp(min=0)
    v[:, :, :2, :2] = 0                                             # an all-zero window: idx 255
    v[:, :, 3, 4] = v[:, :, 3, 5]                                   # exact ties: the first in scan order wins
    v[:, :, 4, 2] = v[:, :, 3, 2]
    v[:, :, 5, 7] = v[:, :, 5, 6] * (1 + 2.0 ** -12)                # same hi, the winner is decided by lo
    hi = v.to(torch.bfloat16).float()
    lo = (v - hi).to(torch.bfloat16).float()
    val = hi + lo                                                   # exact in fp32
    act = torch.cat((tc.nchw_to_pf(hi.to(DEV)), tc.nchw_to_pf(lo.to(DEV))), 1).contiguous()
    oh, ow = h // 2, w // 2
    prow = tc.pf_rows(n, oh, ow)
    pooled = torch.empty(prow, 2 * c, device=DEV, dtype=torch.bfloat16)
    idx = torch.empty(prow, c, device=DEV, dtype=torch.uint8)
    _lib.check(lib.lrpx_tc_maxpool3s2_x(_p(act), _p(pooled), _p(idx), n, h, w, c, 1, _stream()), "maxpool3s2_x")
    ref, iref = F.max_pool2d(val, 3, 2, 1, return_indices=True)
    yy, xx = iref // w, iref % w
    oy, ox = torch.arange(oh).view(1, 1, oh, 1), torch.arange(ow).view(1, 1, 1, ow)
    k_ref = ((yy - (2 * oy - 1)) * 3 + (xx - (2 * ox - 1))).to(torch.uint8)
    zero = ref == 0
    k_ref[zero] = 255
    got_idx = _pf_valid(idx, n, oh, ow, c).cpu()
    assert torch.equal(got_idx, k_ref), "arg-max of hi + lo in PyTorch scan order, 255 where the maximum is 0"
    p = pooled.view(n, oh + 1, ow + 1, 2 * c)[:, 1:, 1:].permute(0, 3, 1, 2).cpu().float()
    want_hi = torch.gather(hi.flatten(2), 2, iref.flatten(2)).view_as(ref).masked_fill(zero, 0.)
    want_lo = torch.gather(lo.flatten(2), 2, iref.flatten(2)).view_as(ref).masked_fill(zero, 0.)
    assert torch.equal(p[:, :c], want_hi) and torch.equal(p[:, c:], want_lo), "pooled keeps the winner's hi|lo row"
    assert torch.equal(p[:, :c] + p[:, c:], ref)
    # split = 0: the bf16 kernel, bit for bit
    a16 = tc.nchw_to_pf(hi.to(DEV))
    p0, i0 = torch.empty(prow, c, device=DEV, dtype=torch.bfloat16), torch.empty(prow, c, device=DEV, dtype=torch.uint8)
    p1, i1 = torch.empty_like(p0), torch.empty_like(i0)
    _lib.check(lib.lrpx_tc_maxpool3s2_x(_p(a16), _p(p0), _p(i0), n, h, w, c, 0, _stream()), "maxpool3s2_x split=0")
    _lib.check(lib.lrpx_tc_maxpool3s2_bf16(_p(a16), _p(p1), _p(i1), n, h, w, c, _stream()), "maxpool3s2")
    torch.cuda.synchronize()
    assert torch.equal(p0, p1) and torch.equal(i0, i1)


# ------------------------------------------------------------------------------------------------ forward and chain
def _nets(golden):
    g = golden("resnet_2111")
    return [("resnet_2111 64x64", g["layers"].tolist(), int(g["seed"]), g["x"], g),
            ("resnet(1,1,1,1) 224x224", [1, 1, 1, 1], 77, torch.randn(1, 3, 224, 224, generator=torch.Generator().manual_seed(78)),
             None)]


@pytest.mark.parametrize("which", [0, 1], ids=["resnet_2111", "resnet1111_224"])
def test_mixed_forward_and_chain_vs_fp64_oracle(golden, which):
    from lrpx import tc_resnet
    name, layers, seed, x, fixture = _nets(golden)[which]
    net = _resnet(layers, seed)
    mixed, bf16 = tc_resnet.TcResNetMixed(net, DEV), tc_resnet.TcResNetEngine(net, DEV)
    assert mixed.precision == "mixed" and not mixed.split
    st, sb = mixed.forward(x.to(DEV)), bf16.forward(x.to(DEV))
    sd64 = {k: (v.double() if v.is_floating_point() else v) for k, v in synth.resnet_state(seed, tuple(layers)).items()}
    gen = torch.Generator().manual_seed(5 + which)
    Q = 5 if which == 0 else 2
    feats = mixed.features(st, "nchw")
    tgt, rimg = _feature_target(feats, gen, Q)
    ref, ref_feats = O.resnet_lrp(sd64, x[rimg.long()].double(), tgt.double(), return_output=True)
    fl2 = max(_rel_l2(feats[i], ref_feats[j]) for j, i in enumerate(rimg.tolist()))
    fl2_bf = max(_rel_l2(bf16.features(sb, "nchw")[i], ref_feats[j]) for j, i in enumerate(rimg.tolist()))
    print(f"{name}: features rel L2 vs fp64: mixed {fl2:.3e}, bf16 {fl2_bf:.3e}")
    assert fl2 <= 1e-4
    assert torch.equal(mixed.features(st, "pixel"), feats.flatten(2).transpose(1, 2))
    heat = mixed.relevance(st, _pix(tgt), rimg.to(DEV), chunk=2)
    heat_bf = bf16.relevance(sb, _pix(tgt), rimg.to(DEV), chunk=2)
    l2s, l2bs = [], []
    for q in range(Q):
        l2, sp = _rel_l2(heat[q], ref[q]), spearman(heat[q].cpu().double(), ref[q])
        l2b = _rel_l2(heat_bf[q], ref[q])
        print(f"{name} request {q} vs fp64 oracle: mixed rel L2 {l2:.3e} spearman {sp:.5f}; bf16 rel L2 {l2b:.3e}")
        assert sp >= 0.99 and l2 <= 6e-2
        l2s.append(l2)
        l2bs.append(l2b)
    assert sum(l2s) <= sum(l2bs), "the accurate forward must not make the heat-maps worse than the bf16 engine's"
    # the chunk size changes no bit in any delivery format; the formats are the full map's channel mean / fp16 rounding
    # (formed in the gather kernel, whose fp32 contractions may fuse differently per format: compared at 1e-5)
    h1 = mixed.relevance(st, _pix(tgt), rimg.to(DEV), chunk=Q)
    assert torch.equal(h1, heat)
    cm = mixed.relevance(st, _pix(tgt), rimg.to(DEV), chunk=3, deliver="channel_mean")
    assert torch.equal(cm, mixed.relevance(st, _pix(tgt), rimg.to(DEV), chunk=Q, deliver="channel_mean"))
    assert_close(cm, h1.mean(1), rtol=1e-5, atol=1e-6 * float(h1.abs().max()), what="channel_mean")
    f16 = mixed.relevance(st, _pix(tgt), rimg.to(DEV), chunk=1, deliver="fp16")
    assert torch.equal(f16, mixed.relevance(st, _pix(tgt), rimg.to(DEV), chunk=Q, deliver="fp16"))
    assert_close(f16.float(), h1, rtol=1e-3, atol=1e-3 * float(h1.abs().max()) + 2.0 ** -24, what="fp16")   # + subnormal step
    if fixture is not None:
        # the fixture's own feature-independent target (see tests/test_gpu_resnet_tc.py::_feature_target): reported
        tf = _pix(fixture["target"])
        hm, hb = mixed.relevance(st, tf), bf16.relevance(sb, tf)
        assert torch.isfinite(hm).all()
        for q in range(x.shape[0]):
            print(f"{name} fixture target request {q} vs the reference's output: mixed rel L2 "
                  f"{_rel_l2(hm[q], fixture['rel'][q]):.3e}, bf16 {_rel_l2(hb[q], fixture['rel'][q]):.3e}")


def test_mixed_accounting_and_fp32_engine(golden):
    from lrpx import tc_resnet, _lib
    g = golden("resnet_2111")
    net = _resnet(g["layers"].tolist(), int(g["seed"]))
    mixed, bf16 = tc_resnet.TcResNetMixed(net, DEV), tc_resnet.TcResNetEngine(net, DEV)
    x = g["x"].to(DEV)
    st, sb = mixed.forward(x), bf16.forward(x)
    assert mixed.heat_shape(3, "channel_mean") == bf16.heat_shape(3, "channel_mean")
    assert mixed.flops_per_explanation() == bf16.flops_per_explanation() == mixed.mma_flops_per_explanation()
    assert mixed.flops_forward_per_image() == 3 * bf16.flops_forward_per_image()
    # the state holds bf16 gains and the hi halves of the block inputs (the chain's operands), like the bf16 engine's
    for gm, gb in zip(st.blocks, sb.blocks):
        for k in gb:
            if torch.is_tensor(gb[k]):
                assert gm[k].dtype == gb[k].dtype and gm[k].shape == gb[k].shape, k
    fp32 = tc_resnet.TcResNetEngine(net, DEV, precision="fp32")
    s32 = fp32.forward(x)
    assert torch.equal(fp32.features(s32), mixed.features(st))
    with pytest.raises(_lib.LrpxError):
        fp32.relevance(s32, torch.zeros(x.shape[0], s32.feat_hw[0] * s32.feat_hw[1], s32.feat_c, device=DEV))


# ------------------------------------------------------------------------------------------------ routes
def _args(E, H, tmp_path):
    return argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="resnet101", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")


def _gridtd_resnet101(V, H, E):
    from models import gridTDmodel as G
    torch.manual_seed(23)
    model = G.GridTDModel(E, H, V, "resnet101", n_pixel=49)
    model.load_state_dict(synth.gridtd_decoder_state(331, V, H, E, C=2048, n_pixel=49), strict=False)
    return model.to(DEV).eval()


def test_compute_lrp_and_explainers_route_mixed(golden, tmp_path):
    from LRPtools import lrp_wrapper
    from lrpx import _lib
    g = golden("resnet_2111")
    net = _resnet(g["layers"].tolist(), int(g["seed"]))
    lrp_wrapper.add_lrp(net)
    x = g["x"].to(DEV)
    _, feats = net.compute_lrp(x.clone(), target=g["target"].to(DEV), return_output=True)
    tgt = g["target"].to(DEV) * feats
    before = dict(_lib.CALLS)
    rm, fm = net.compute_lrp(x.clone(), target=tgt, precision="mixed", return_output=True)
    for k in ("lrpx_tc_im2col7s2_split_x", "lrpx_tc_maxpool3s2_x", "lrpx_tc_conv"):
        assert _lib.CALLS.get(k, 0) > before.get(k, 0), k
    r32 = net.compute_lrp(x.clone(), target=tgt, precision="simt")
    print(f"compute_lrp mixed vs simt: rel L2 {_rel_l2(rm, r32):.3e}, spearman {spearman(rm.cpu().double(), r32.cpu().double()):.5f}")
    assert spearman(rm.cpu().double(), r32.cpu().double()) >= 0.99
    assert_close(fm, feats, rtol=1e-4, atol=1e-4 * float(feats.abs().max()), what="features")
    for m in net.modules():
        if hasattr(m, "lrp_params"):
            m.lrp_params = dict(m.lrp_params, alpha=2., beta=1.)
    with pytest.raises(NotImplementedError):
        net.compute_lrp(x.clone(), target=tgt, precision="mixed")
    from models import gridTDmodel as G
    from models import adaptiveattention as A
    V, H, E = 60, 64, 32
    ex = G.ExplainGridTDAttention(_args(E, H, tmp_path), synth.word_map(V), model=_gridtd_resnet101(V, H, E),
                                  precision="mixed")
    assert ex.uses_tc and ex.is_resnet
    am = A.AdaptiveAttentionCaptioningModel(H, H, V, "resnet101", n_pixel=49).to(DEV).eval()
    ea = A.ExplainAdaptiveAttention(_args(H, H, tmp_path), synth.word_map(V), model=am, precision="mixed")
    assert ea.uses_tc and ea.is_resnet
    with pytest.raises(NotImplementedError):
        G.ExplainGridTDGradient(_args(E, H, tmp_path), synth.word_map(V), model=ex.model, precision="mixed")


# ------------------------------------------------------------------------------------------------ explainers
def test_explain_caption_resnet101_mixed_vs_simt(tmp_path):
    from models import gridTDmodel as G
    V, H, E = 60, 64, 32
    model = _gridtd_resnet101(V, H, E)
    img = synth.images(332, 1).to(DEV)
    toks = synth.tokens(333, 2, V)
    outs = {}
    for prec in ("simt", "mixed", "bf16"):
        ex = G.ExplainGridTDAttention(_args(E, H, tmp_path), synth.word_map(V), model=model, precision=prec)
        ex.ACCUMULATE_LIKE_REFERENCE = False
        ex.preprocess_img = lambda p: img
        model.beam_search = lambda *a, **k: (["a b"], toks[1:])
        outs[prec] = ex.explain_caption("synthetic.jpg")
    for t in range(2):
        hs, ws = outs["simt"][0][t], outs["simt"][1][t]
        hm, wm = outs["mixed"][0][t], outs["mixed"][1][t]
        hb, wb = outs["bf16"][0][t], outs["bf16"][1][t]
        sp = spearman(hm.cpu().double(), hs.cpu().double())
        print(f"word {t}: mixed vs simt words max err {float((wm - ws).abs().max()):.3e} (bf16 "
              f"{float((wb - ws).abs().max()):.3e}); heat-map spearman {sp:.5f}, rel L2 {_rel_l2(hm, hs):.3e} "
              f"(bf16 {_rel_l2(hb, hs):.3e})")
        assert_close(wm, ws, rtol=1e-3, atol=1e-3, what=f"mixed r_words t={t}")
        assert sp >= 0.99


def test_batch_explainer_on_mixed_resnet(tmp_path):
    from models import gridTDmodel as G
    from lrpx.pipeline import BatchExplainer
    V, H, E, B, T = 60, 64, 32, 2, 3
    model = _gridtd_resnet101(V, H, E)
    ex = G.ExplainGridTDAttention(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="mixed")
    ex.ACCUMULATE_LIKE_REFERENCE = False
    imgs = synth.images(313, B).to(DEV)
    toks = torch.tensor([synth.tokens(314 + b, T, V) for b in range(B)], device=DEV)
    heat, r_words = BatchExplainer(ex, chunk=4).explain(imgs, toks)
    heat, r_words = heat.clone(), r_words.clone()
    heat_g, words_g = BatchExplainer(ex, chunk=4, use_graph=True).explain(imgs, toks)
    assert torch.equal(heat_g, heat) and torch.equal(words_g, r_words), "graph replay"
    for b in range(B):
        ex.img = imgs[b:b + 1]
        ex.beam_caption_encode = toks[b].tolist()
        ex._set_state(ex.img, ex.beam_caption_encode)
        for t in (0, T - 1):
            r_img, rw = ex.explain_caption_wordt(t)
            one = ex.explain_cnn(r_img)
            q = b * T + t
            assert_close(heat[q:q + 1], one, rtol=1e-3, atol=1e-4 * float(one.abs().max()), what=f"image {b} word {t}")
            assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=1e-5, what=f"words image {b} word {t}")


def test_mixed_explainer_after_bn_update_equals_fresh(tmp_path):
    from models import gridTDmodel as G
    V, H, E = 60, 64, 32
    model = _gridtd_resnet101(V, H, E)
    img = synth.images(95, 1).to(DEV)
    tk = synth.tokens(96, 3, V)

    def run(ex):
        ex.preprocess_img = lambda p: img
        ex.model.beam_search = lambda *a, **k: (["w1 w2 w3"], tk[1:])
        ex.ACCUMULATE_LIKE_REFERENCE = False
        heat, words = ex.explain_caption("synthetic.jpg")
        return torch.cat(heat), [w.clone() for w in words]

    make = lambda: G.ExplainGridTDAttention(_args(E, H, tmp_path), synth.word_map(V), model=model, precision="mixed")
    ex = make()
    before = run(ex)
    with torch.no_grad():
        model.img_encoder.encoder.layer1[0].bn2.running_var.mul_(1.7)
    after, fresh = run(ex), run(make())
    assert not torch.equal(before[0], fresh[0]), "the update did not change the explanation"
    assert torch.equal(after[0], fresh[0])
    for a, f in zip(after[1], fresh[1]):
        assert torch.equal(a, f)
