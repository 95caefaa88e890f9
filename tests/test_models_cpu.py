"""CPU: host-side logic of the model mirrors — state_dict compatibility with the reference layout, the
explainer's teacher-forced forward (incl. quirks Q3/Q19) against the reference fixtures, beam search."""
import argparse

import pytest
import torch

import lrp_oracle as O
import synth
from conftest import assert_close


def _explainer(g, tmp_path):
    from models import gridTDmodel as G
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    model = G.GridTDModel(E, H, V, "vgg16")
    sd = synth.gridtd_decoder_state(int(g["seed"]), V, H, E)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith("img_encoder.") for k in missing)
    args = argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")
    return G.ExplainGridTDAttention(args, synth.word_map(V), model=model), sd


@pytest.mark.parametrize("name", ["gridtd_dec_small", "gridtd_dec_512"])
def test_explainer_forward_matches_reference_fixture(golden, tmp_path, name):
    """The tensor-op restatement in tests/helpers.py (the checker of the fused CUDA explainer forward, see
    tests/test_gpu_models.py) against the reference's own get_hidden_parameters outputs; the product method
    itself refuses CPU tensors."""
    import helpers
    from lrpx._lib import LrpxError
    g = golden(name)
    ex, sd = _explainer(g, tmp_path)
    feat = g["feats"][0].flatten(1).t().unsqueeze(0).contiguous()          # (1,P,C)
    toks = torch.tensor([g["tokens"].tolist()])
    with pytest.raises(LrpxError):
        ex.explainer_forward(feat, toks)
    st = helpers.gridtd_explainer_forward_ops(ex.model, feat, toks)
    assert_close(st["pred"][0], g["predictions"], atol=3e-5, what="predictions")
    assert_close(st["alpha"][0], g["alphas"].reshape(st["alpha"][0].shape), atol=1e-6, what="alphas")
    assert_close(st["beta"][0], g["betas"].reshape(-1), atol=1e-6, what="betas")
    assert_close(st["h2"][0], g["h2t"], atol=1e-5, what="h2t")
    assert_close(st["c1"][0], g["c1t"], atol=1e-5, what="c1t")
    assert_close(st["ctx_hat"][0], g["context_hat"], atol=1e-5, what="context_hat")
    # and key-by-key against the oracle's restatement
    ost = O.gridtd_explainer_forward(sd, g["feats"][0], g["tokens"].tolist())
    for k, ok in [("x1", "x1"), ("x2", "x2"), ("g1", "g1"), ("i2", "i2"), ("st", "s"), ("ctx", "ctx"), ("A_pre", "A_pre")]:
        assert_close(st[k][0], ost[ok], atol=2e-5, what=k)


def test_state_dict_keys_match_reference_layout():
    from models import gridTDmodel as G, vgg, resnet
    m = G.GridTDModel(32, 48, 50, "vgg16")
    keys = set(k for k in m.state_dict() if not k.startswith("img_encoder."))
    assert keys == set(synth.gridtd_decoder_state(0, 50, 48, 32).keys())
    enc_keys = set(k[len("img_encoder.encoder."):] for k in m.state_dict() if k.startswith("img_encoder.encoder."))
    assert enc_keys == set(synth.vgg_state(0).keys())
    r = resnet.ResNet(resnet.Bottleneck, [2, 1, 1, 1])
    assert set(r.state_dict().keys()) == set(synth.resnet_state(0, (2, 1, 1, 1)).keys())


def test_beam_search_runs_and_uses_floor_division():
    from models import gridTDmodel as G
    torch.manual_seed(0)
    V = 40
    m = G.GridTDModel(16, 24, V, "vgg16").eval()
    wm = synth.word_map(V)
    sent, idx = m.beam_search(torch.randn(1, 3, 224, 224), wm, beam_size=2, max_cap_length=6)
    assert isinstance(sent, list) and all(0 < i < V - 3 for i in idx) and len(idx) <= 20


def test_lrp_linear_eps_has_no_cpu_form():
    """The named vector rule is a CUDA entry point (lrpx_lrp_linear_eps_f32; parity in tests/test_gpu_rules.py): on
    CPU tensors it raises instead of falling back to a tensor expression."""
    from models import gridTDmodel as G
    from lrpx._lib import LrpxError
    m = G.GridTDModel(8, 8, 20, "vgg16")
    g = torch.Generator().manual_seed(1)
    x, w, r = torch.randn(6, generator=g), torch.randn(5, 6, generator=g), torch.randn(5, generator=g)
    with pytest.raises(LrpxError):
        m.lrp_linear_eps(r, x, w @ x, w)


@pytest.mark.parametrize("name", ["aoa_dec_512", "aoa_dec_bu"])
def test_aoa_explainer_forward_matches_reference_fixture(golden, tmp_path, name):
    from models import aoamodel as A
    g = golden(name)
    V, H, E, C = int(g["V"]), int(g["H"]), int(g["E"]), int(g["C"])
    model = A.AOAModel(E, H, 8, V, "vgg16")
    model.img_projector = torch.nn.Conv2d(C, H, 1)
    model.encoder_raw_dim = C
    sd = synth.aoa_decoder_state(int(g["seed"]), V, H, E, C)
    missing, unexpected = model.load_state_dict(sd, strict=False)
    assert not unexpected and all(k.startswith("img_encoder.") for k in missing)
    args = argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")
    ex = A.ExplainAOAAttention(args, synth.word_map(V), model=model)
    feat = g["feats"][0].flatten(1).t().unsqueeze(0).contiguous()
    import helpers
    from lrpx._lib import LrpxError
    with pytest.raises(LrpxError):                       # the product's forward is CUDA only
        ex.explainer_forward(feat, torch.tensor([g["tokens"].tolist()]))
    st = helpers.aoa_explainer_forward_ops(ex.model, feat, torch.tensor([g["tokens"].tolist()]))
    assert_close(st["pred"][0], g["predictions"], atol=5e-5, what="predictions")
    assert_close(st["alpha"][0], g["alphas"].reshape(st["alpha"][0].shape), atol=1e-6, what="alphas")
    assert_close(st["h"][0], g["ht"], atol=1e-5, what="ht")
    assert_close(st["caoa"][0], g["context_aoa"], atol=1e-5, what="context_aoa")
    with pytest.raises(LrpxError):                       # lrp_mha is a CUDA entry point too (tests/test_gpu_rules.py)
        ex.lrp_mha(st["alpha"][0, 0], st["value"][0], st["ctx"][0, :1], st["ctx"][0, :1], 0)


def _bu_models(g):
    """The bottom-up twins with the fixture's synthetic weights (incl. its <end> bias)."""
    from models import gridTDmodel as G, aoamodel as A
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    s = g["seeds"].tolist()
    out = {}
    for tag, m, sd in (("gridtd", G.GridTDModelBU(E, H, V, "bu"), synth.gridtd_bu_state(s[0], V, H, E)),
                       ("aoa", A.AOAModelBU(E, H, 8, V, "bu"), synth.aoa_bu_state(s[1], V, H, E))):
        sd["fc.bias"][V - 1] += float(g["end_bias"])
        m.load_state_dict(sd, strict=True)          # key-for-key the reference's state_dict layout
        out[tag] = m.eval()
    return out, V, s


def test_bu_beam_search_indices_bit_exact_vs_reference(golden):
    """AOAModelBU / GridTDModelBU.beam_search on 36 x 2048 region features (BASELINE config 3: beam size 3): the
    word indices must equal the reference's own output bit for bit (finished and unfinished beams both occur)."""
    g = golden("tune_bu")
    models, V, s = _bu_models(g)
    wm = synth.word_map(V)
    feats = synth.bu_features(s[2], 3)
    for tag, m in models.items():
        ref = g[f"{tag}_beams"]
        row = 0
        for b in range(3):
            for bs in (1, 3):
                _, sen_idx = m.beam_search(feats[b:b + 1], wm, beam_size=bs)
                want = [int(v) for v in ref[row] if int(v) >= 0]
                assert sen_idx == want, (tag, b, bs, sen_idx, want)
                row += 1


def test_adaptive_model_state_dict_and_search_bit_exact_vs_reference(golden):
    """SURVEY §8 f2: the AdaptiveAttentionCaptioningModel mirror loads the reference's state_dict layout key for key,
    and its beam_search (beam sizes 1 and 3) / greedy_search reproduce the reference's word indices bit for bit
    (adaptiveattention.py:370-489; finished and unfinished beams both occur in the fixture)."""
    from models import adaptiveattention as AA
    g = golden("adaptive_dec_small")
    V, H, E, seed = int(g["V"]), int(g["H"]), int(g["E"]), int(g["seed"])
    m = AA.AdaptiveAttentionCaptioningModel(E, H, V, "vgg16")
    sd = synth.adaptive_decoder_state(seed, V, H, E)
    assert set(k for k in m.state_dict() if not k.startswith("img_encoder.")) == set(sd.keys())
    sd["fc.bias"][V - 1] += float(g["end_bias"])
    m.load_state_dict(sd, strict=False)
    m.eval()
    wm = synth.word_map(V)

    class Stub(torch.nn.Module):
        def __init__(self, f):
            super().__init__()
            self.f = f

        def forward(self, img):
            return self.f, self.f.mean((2, 3)).squeeze()

    row = 0
    for b in range(3):
        gen = torch.Generator().manual_seed(seed + 10 + b)
        m.img_encoder = Stub(torch.randn(1, 512, 14, 14, generator=gen).clamp(min=0))
        for bs in (1, 3):
            _, sen_idx = m.beam_search(torch.zeros(1, 3, 224, 224), wm, beam_size=bs)
            want = [int(v) for v in g["beams"][row] if int(v) >= 0]
            assert sen_idx == want, (b, bs, sen_idx, want)
            row += 1
        _, seqs = m.greedy_search(torch.zeros(1, 3, 224, 224), wm, max_cap_length=12)
        assert seqs[0] == g["greedy"][b].tolist(), (b, seqs[0], g["greedy"][b].tolist())


def test_adaptive_explainer_refuses_cpu(tmp_path):
    from models import adaptiveattention as AA
    from lrpx._lib import LrpxError
    V, H = 50, 32
    m = AA.AdaptiveAttentionCaptioningModel(H, H, V, "vgg16")
    args = argparse.Namespace(embed_dim=H, hidden_dim=H, encoder="vgg16", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")
    ex = AA.ExplainAdaptiveAttention(args, synth.word_map(V), model=m)
    with pytest.raises(LrpxError):
        ex.explainer_forward(torch.zeros(1, 196, 512), torch.zeros(1, 4, dtype=torch.long))
    with pytest.raises(ValueError):
        AA.ExplainAdaptiveAttention(args, synth.word_map(V), model=AA.AdaptiveAttentionCaptioningModel(16, H, V, "vgg16"))


def test_sample_greedy_matches_reference_and_reward_criterion(golden):
    """GridTDModel.sample (the greedy baseline of trainciderlrp, train.py:259-261) on the full VGG16 model against the
    reference's own output; RewardCriterion (modelutils.py:31-46) against its formula."""
    from models import gridTDmodel as G
    from lrpx.tune import RewardCriterion
    g = golden("tune_gridtd")
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    s = g["seeds"].tolist()
    m = G.GridTDModel(E, H, V, "vgg16")
    m.load_state_dict(synth.gridtd_decoder_state(s[0], V, H, E), strict=False)
    m.img_encoder.encoder.load_state_dict(synth.vgg_state(s[1]))
    m.eval()
    with torch.no_grad():
        seq, lp, L = m.sample(synth.images(s[2], 2), synth.word_map(V), torch.tensor([9, 9]))
    assert L == 8 and torch.equal(seq, g["sample_seq"])
    assert_close(lp, g["sample_logprobs"], atol=1e-4, what="sample logprobs")
    gen = torch.Generator().manual_seed(5)
    logp = -torch.rand(3, 6, generator=gen)
    seqs = torch.tensor([[4, 7, 0, 0, 0, 0], [3, 3, 3, 3, 3, 3], [0, 0, 0, 0, 0, 0]])
    reward = torch.randn(3, 1, generator=gen).expand(3, 6)
    mask = torch.tensor([[1., 1, 1, 0, 0, 0], [1, 1, 1, 1, 1, 1], [1, 0, 0, 0, 0, 0]])
    want = (-logp * reward * mask).sum() / mask.sum()
    assert_close(RewardCriterion()(logp, seqs, reward), want, what="reward criterion")


def test_adaptive_model_forward_matches_reference(golden):
    """AdaptiveAttentionCaptioningModel.forward (teacher forcing, adaptiveattention.py:137-190) against the reference's
    own predictions / alphas / betas on two stubbed feature maps."""
    from models import adaptiveattention as AA
    g = golden("adaptive_dec_small")
    V, H, E, seed = int(g["V"]), int(g["H"]), int(g["E"]), int(g["seed"])
    m = AA.AdaptiveAttentionCaptioningModel(E, H, V, "vgg16")
    sd = synth.adaptive_decoder_state(seed, V, H, E)
    sd["fc.bias"][V - 1] += float(g["end_bias"])
    m.load_state_dict(sd, strict=False)
    m.eval()
    fb = torch.cat([torch.randn(1, 512, 14, 14, generator=torch.Generator().manual_seed(seed + 10 + b)).clamp(min=0)
                    for b in range(2)])

    class Stub(torch.nn.Module):
        def forward(self, img):
            return fb, fb.mean((2, 3)).squeeze()

    m.img_encoder = Stub()
    with torch.no_grad():
        pred, alphas, betas, _, L = m(torch.zeros(2, 3, 224, 224), g["fwd_caps"], torch.tensor([5, 4]), None)
    assert L == int(g["fwd_max_length"])
    assert_close(pred, g["fwd_predictions"], atol=2e-5, what="forward predictions")
    assert_close(alphas, g["fwd_alphas"], atol=1e-6, what="forward alphas")
    assert_close(betas, g["fwd_betas"], atol=1e-6, what="forward betas")


def test_bu_twins_forward_and_greedy_sample_vs_reference(golden):
    """GridTDModelBU / AOAModelBU: the plain teacher-forced ``forward`` and the greedy ``sample`` (the self-critical
    baseline of trainciderlrp) against the reference's own outputs — logits to 2e-5, sampled words bit-exact."""
    g = golden("tune_bu")
    models, V, s = _bu_models(g)
    wm = synth.word_map(V)
    feats = synth.bu_features(s[2], 3)
    for tag, m in models.items():
        with torch.no_grad():
            pred = m(feats, g["caps"], g["caplens"], None)[0]
            seq, lp, _ = m.sample(feats, wm, g["caplens"])
        assert_close(pred, g[f"{tag}_fwd_predictions"], atol=2e-5, what=f"{tag} forward")
        assert torch.equal(seq, g[f"{tag}_sample_seq"]), tag
        assert_close(lp, g[f"{tag}_sample_logprobs"], atol=1e-4, what=f"{tag} sample logprobs")


def test_encoder_mirrors_forward_vs_reference_fixtures(golden):
    """models.resnet.ResNet and models.vgg (features[0:-1]) mirrors: forward on the fixtures' inputs equals the
    reference's encoder output (state_dict-compatible modules, plain torch forward)."""
    from models import resnet, vgg
    g = golden("resnet_2111")
    r = resnet.ResNet(resnet.Bottleneck, g["layers"].tolist())
    r.load_state_dict(synth.resnet_state(int(g["seed"]), tuple(g["layers"].tolist())))
    r.eval()
    with torch.no_grad():
        assert_close(r(g["x"]), g["feats"], atol=2e-5, what="resnet mirror forward")
    g = golden("vgg16_64")
    enc = vgg.vgg16(pretrained=False).features[0:-1]
    enc.load_state_dict(synth.vgg_state(int(g["seed"])))
    enc.eval()
    with torch.no_grad():
        assert_close(enc(g["x"]), g["feats"], atol=2e-5, what="vgg mirror forward")


def test_heatmap_postprocessing_matches_reference_fixture(golden):
    """LRPtools.utils.project / gamma (utils.py:34-52,101-145) against values the reference's own functions produced
    (fixture utils_viz, generated through oracle/ref_shim.py); heatmap's colour tables: 'seismic' runs dark blue - blue -
    white - red - dark red, 'gray' black - white, 256 entries like matplotlib's."""
    import numpy as np
    import LRPtools.utils as U
    g = golden("utils_viz")
    x = g["x"].numpy()
    assert np.array_equal(U.project(x.copy()), g["proj"].numpy())
    assert np.array_equal(U.project(x.copy(), output_range=(0, 255)), g["proj255"].numpy())
    assert np.allclose(U.gamma(x.copy(), 0.7), g["gamma"].numpy(), rtol=1e-6, atol=1e-7)
    lut = U._CMAPS["seismic"]
    assert lut.shape == (256, 3) and np.allclose(lut[0], (0, 0, 0.3)) and np.allclose(lut[-1], (0.5, 0, 0))
    assert np.allclose(lut[127], lut[128][::-1], atol=2e-2) and lut[127:129].min() > 0.98          # white in the middle
    hm = U.heatmap(np.stack([x[0]] * 3, -1)[None])                         # (1,16,16,3) -> RGB
    assert hm.shape == (1, 16, 16, 3) and hm.dtype == np.float32
    gm = U.graymap(np.stack([x[0]] * 3, -1)[None])
    assert np.allclose(gm[..., 0], gm[..., 1]) and np.allclose(gm[..., 1], gm[..., 2])


def test_tpfp_split_host_logic(golden):
    """lrpx.ablation.AblationExperiments.tpfp_split (evaluation.py:462-481,:516) against the reference's own TP / FP
    filing recorded in fixture ablation_e2e."""
    from lrpx.ablation import AblationExperiments
    g = golden("ablation_e2e")
    V = int(g["V"])
    wm = synth.word_map(V)
    toks = g["tokens"].tolist()
    frequent = [i for w, i in wm.items() if w.startswith("w")]
    special = [wm[k] for k in ("<start>", "<pad>", "<end>", "<unk>")]
    tp, fp = AblationExperiments.tpfp_split(toks, frequent, [g["ref_caps_0"].tolist(), g["ref_caps_1"].tolist()], special)
    assert [toks[t + 1] for t in tp] == g["tp_words"].tolist() and [toks[t + 1] for t in fp] == g["fp_words"].tolist()
    assert AblationExperiments.tpfp_split(toks, [], [toks], special) == ([], [])


def test_expand_operator_matches_scipy():
    """models/_gradient.py::expand_operator (pyramid_expand along one axis as a matrix) against the same two steps done
    with scipy: bilinear interpolation at (r + 0.5)/16 - 0.5 with mirrored borders, then gaussian_filter(sigma = 16/3,
    mode='reflect').  (skimage, whose pyramid_expand this restates, is not installed: parity unpinned.)"""
    import numpy as np
    from scipy import ndimage
    from models._gradient import expand_operator
    rng = np.random.default_rng(5)
    cam = rng.random((14, 14))
    K = expand_operator(14, 16)
    assert K.shape == (224, 14) and np.allclose(K.sum(1), 1.0)
    coords = (np.arange(224) + 0.5) / 16 - 0.5
    yy, xx = np.meshgrid(coords, coords, indexing="ij")
    resized = ndimage.map_coordinates(cam, [yy, xx], order=1, mode="mirror")
    want = ndimage.gaussian_filter(resized, sigma=2 * 16 / 6.0, mode="reflect")
    got = K @ cam @ K.T
    assert np.abs(got - want).max() < 1e-12


def test_gradient_family_classes_mirror_the_reference_names():
    from models import gridTDmodel as G, aoamodel as A
    for mod, names in ((G, ["ExplainGridTDGradient", "ExplainiGridTDGuidedGradient", "ExplainGridTDGradCam",
                            "ExplainGridTDGuidedGradCam"]),
                       (A, ["ExplainAOAGradient", "ExplainAOAGuidedGradient", "ExplainAOAGradCam", "ExplainAOAGuidedGradCam"])):
        for n in names:
            cls = getattr(mod, n)
            for meth in ("get_hidden_parameters", "explain_caption_wordt", "explain_cnn", "explain_caption",
                         "teacherforce_forward"):
                assert callable(getattr(cls, meth)), (n, meth)
    assert G.ExplainGridTDGuidedGradCam.EX_TYPE == "GuidedGradCam" and A.ExplainAOAGradCam.EX_TYPE == "GradCam"


def test_self_critical_reward_vs_reference_fixture(golden):
    """models/modelutils.get_self_critical_reward (own CIDEr / BLEU restatement in lrpx.scst) and RewardCriterion vs
    the reference's own functions with its vendored pycocoevalcap scorers (fixture scst_reward): CIDEr only (the
    training setting), BLEU only, and a weighted mix."""
    import numpy as np
    import torch
    from models import modelutils as mu
    g = golden("scst_reward")
    wm = synth.word_map(int(g["V"]))
    gen, greedy, gts = g["gen"], g["greedy"], g["gts"]
    data_gts = [[gts[b, r].numpy() for r in range(gts.shape[1])] for b in range(gts.shape[0])]
    for tag, (cw, bw) in {"cider": (1.0, 0.0), "bleu": (0.0, 1.0), "mix": (0.7, 0.3)}.items():
        got = mu.get_self_critical_reward(greedy, data_gts, gen, wm, cw, bw)
        want = g["reward_" + tag].numpy()
        assert got.shape == want.shape and got.dtype == np.float64
        assert np.abs(got - want).max() <= 1e-12 * max(1.0, np.abs(want).max()), tag
        assert np.abs(want).max() > 0.05
    assert float(got[0].max()) == 0.0                      # identical sampled and greedy captions: no advantage
    loss = mu.RewardCriterion()(g["logp"], gen, torch.from_numpy(g["reward_cider"].numpy()).float())
    assert abs(float(loss) - float(g["loss"])) <= 1e-6 * abs(float(g["loss"]))
    rev = {v: k for k, v in wm.items()}
    s = mu.array_to_str(gen[2].tolist(), rev, wm['<end>'])
    assert '<start>' not in s and '<pad>' not in s


def test_greedy_search_equals_beam_size_one():
    """GridTDModel / AOAModel.greedy_search (reference gridTDmodel.py:480-520, aoamodel.py:487-530): for one image the
    words are those of beam_search with one beam (what the explainers' forward_greedy runs), until <end>."""
    import torch
    from models import gridTDmodel as G, aoamodel as A
    V, H, E = 40, 32, 16
    wm = synth.word_map(V)
    torch.manual_seed(3)
    for model in (G.GridTDModel(E, H, V, "vgg16"), A.AOAModel(E, H, 4, V, "vgg16")):
        model.eval()
        img = synth.images(4, 1)
        sent_b, idx_b = model.beam_search(img, wm, beam_size=1, max_cap_length=8)
        sent_g, seqs = model.greedy_search(img, wm, max_cap_length=8)
        special = {wm['<start>'], wm['<end>'], wm['<unk>'], wm['<pad>']}
        words_g = [w for w in seqs[0] if w not in special]
        words_b = [w for w in idx_b if w not in special]
        n = min(len(words_g), len(words_b))
        assert n > 0 and words_g[:n] == words_b[:n], (words_g, words_b)
        assert seqs[0][0] == wm['<start>'] and len(seqs[0]) == 8 and isinstance(sent_g[0], str)


def test_decoder_workspace_cache_policy(monkeypatch):
    """ops._decoder_workspace (host logic, no GPU): a workspace is kept per argument shape only for the tensor-core GEMM
    mode, is handed back with LRPX_DEC_W3_READY on the next call of that shape, is stored by the caller only AFTER a
    successful call, never during a stream capture, and at most four shapes are kept (nothing is ever evicted: a captured
    graph may point into an entry)."""
    import torch
    from lrpx import ops
    made = []

    def fake_empty(n, device=None, dtype=None):
        made.append(n)
        return ("ws", len(made))

    capturing = {"on": False}
    monkeypatch.setattr(torch, "empty", fake_empty)
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: capturing["on"])
    cache = {}
    ws, extra, key = ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True)
    assert extra == 0 and key == ("gridtd", (1, 2, 3), 100) and cache == {}       # miss: the caller stores it after the call
    cache[key] = ws
    ws2, extra2, key2 = ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True)
    assert ws2 is ws and extra2 == ops.DEC_W3_READY and key2 is None
    # another shape / another decoder: another entry
    _, e3, k3 = ops._decoder_workspace(cache, "gridtd", (1, 2, 4), 100, "cuda", True)
    _, e4, k4 = ops._decoder_workspace(cache, "aoa", (1, 2, 3), 100, "cuda", True)
    assert e3 == 0 and e4 == 0 and k3 != key and k4 != key and k3 != k4
    # fp32 CUDA-core GEMMs, no cache dict, or a running capture: a fresh workspace that is not kept
    assert ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", False)[1:] == (0, None)
    assert ops._decoder_workspace(None, "gridtd", (1, 2, 3), 100, "cuda", True)[1:] == (0, None)
    capturing["on"] = True
    assert ops._decoder_workspace(cache, "gridtd", (9, 9, 9), 100, "cuda", True)[1:] == (0, None)
    assert ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True)[1] == ops.DEC_W3_READY   # a hit is fine
    capturing["on"] = False
    # the cap: four shapes
    for i in range(3):
        _, _, k = ops._decoder_workspace(cache, "gridtd", (7, i), 100, "cuda", True)
        assert k is not None
        cache[k] = ("ws", i)
    assert len(cache) == 4
    assert ops._decoder_workspace(cache, "gridtd", (8, 8), 100, "cuda", True)[1:] == (0, None)
    assert ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 0, "cuda", True)[0] is not None            # nbytes 0 -> 4-byte dummy
    assert made[-1] == 4


def test_decoder_workspace_cache_keyed_on_weights(monkeypatch):
    """ops._decoder_workspace with the call's weights (host logic, no GPU): the prepared weight copies in a cached
    workspace belong to the weights they were made from.  Other weight tensors of the same shapes, or the same tensors
    after an in-place update (a new version counter, even when the values come back), are another entry."""
    import torch
    from lrpx import ops
    W = {"W_b": torch.zeros(3), "W_a": torch.zeros(2)}
    W2 = {"W_b": torch.zeros(3), "W_a": torch.zeros(2)}
    monkeypatch.setattr(torch, "empty", lambda n, device=None, dtype=None: ("ws", n))
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: False)
    cache = {}
    ws, extra, key = ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True, W)
    assert extra == 0 and key is not None
    cache[key] = ws
    assert ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True, W)[1] == ops.DEC_W3_READY
    assert ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True, dict(reversed(W.items())))[1] == \
        ops.DEC_W3_READY                                                  # the key does not depend on the dict's order
    _, e2, k2 = ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True, W2)
    assert e2 == 0 and k2 not in (None, key)
    W["W_a"].add_(1.0)
    W["W_a"].sub_(1.0)
    _, e3, k3 = ops._decoder_workspace(cache, "gridtd", (1, 2, 3), 100, "cuda", True, W)
    assert e3 == 0 and k3 not in (None, key, k2)
