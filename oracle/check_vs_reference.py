"""The oracle against the UNMODIFIED original project (SunJiamei/LRP-imagecaptioning-pytorch) on cases of its own (fresh
seeds and shapes that the fixtures of make_golden.py do not use): compute_lrp on a non-square conv/relu/max-pool stack,
get_lrp_weight_step, ExplainAdaptiveAttention, and evaluation.py's block_image and bbox share.

  python oracle/check_vs_reference.py          the original executed live through ref_shim, compared with the oracle and
                                               with tests/golden/live_check.npz; exit status 0 = every comparison within
                                               its bar, 77 = the original is not available
  python oracle/check_vs_reference.py --store  writes tests/golden/live_check.npz: the cases' inputs and the expected
                                               outputs — the original's where it is available, else the oracle's (the
                                               file's `source` says which)

tests/test_oracle_vs_reference.py compares the oracle with the stored outputs in every run, and runs this script where the
original is available.  Run as a script: the original's package names `models`, `LRPtools` collide with the product's
mirrors of the same names."""
import contextlib
import io
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import lrp_oracle as O  # noqa: E402
import ref_shim  # noqa: E402
import synth  # noqa: E402

FIXTURE = os.path.join(ROOT, "tests", "golden", "live_check.npz")
CFG = [8, "M", 16, 16, "M", 24]                         # conv/relu/max-pool stack, weights synth.vgg_state(101, CFG)
LW = dict(V=90, H=48, E=16, B=5)                        # get_lrp_weight_step, weights synth.gridtd_decoder_state(103, ...)
ADA = dict(V=200, H=48, T=5)                            # ExplainAdaptiveAttention, weights synth.adaptive_decoder_state(105, ...)
BOXES = [[10, 5, 60, 40], [0, 0, 96, 64], [30, 30, 31, 64]]
THRESHOLDS = [0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9]
PATCHES, PATCH = 20, 8                                  # EvaluationExperiments.num_delete_patches / patch_size
# output -> (rtol, atol); adaptive_r_feat is compared after dividing both sides by the largest |expected| value
BARS = {"conv_stack_rel": (1e-4, 1e-6), "w_ctx": (1e-4, 1e-5), "w_h": (1e-4, 1e-5), "adaptive_pred": (1e-4, 2e-5),
        "adaptive_r_feat": (1e-3, 1e-5), "adaptive_r_words": (1e-3, 1e-5), "block_mask": (1e-4, 0.0),
        "bbox_share": (1e-4, 1e-5)}


def case_inputs():
    g = torch.Generator().manual_seed(102)
    conv_x, conv_target = torch.randn(2, 3, 24, 16, generator=g), torch.randn(2, 24, 6, 4, generator=g)
    g = torch.Generator().manual_seed(104)
    B, V, H = LW["B"], LW["V"], LW["H"]
    logits, h, c = torch.randn(B, V, generator=g), torch.randn(B, H, generator=g), torch.randn(B, H, generator=g)
    feats = torch.randn(1, 512, 14, 14, generator=torch.Generator().manual_seed(106)).clamp(min=0)
    heat = torch.randn(1, 3, 64, 96, generator=torch.Generator().manual_seed(108))
    return {"conv_x": conv_x, "conv_target": conv_target, "logits": logits, "h": h, "c": c, "adaptive_feats": feats,
            "adaptive_tokens": torch.tensor(synth.tokens(107, ADA["T"], ADA["V"])), "heat": heat}


def oracle_outputs(inp):
    out = {"conv_stack_rel": O.sequential_lrp(O.vgg_layers_from_state(synth.vgg_state(101, CFG), CFG), inp["conv_x"],
                                              inp["conv_target"])}
    dsd = synth.gridtd_decoder_state(103, LW["V"], LW["H"], LW["E"])
    out["w_ctx"], out["w_h"] = O.lrp_weight_step(inp["logits"], inp["h"], inp["c"], dsd["fc.weight"],
                                                 synth.stop_mask(LW["V"]))
    asd = synth.adaptive_decoder_state(105, ADA["V"], ADA["H"], ADA["H"])
    st = O.adaptive_explainer_forward(asd, inp["adaptive_feats"][0], inp["adaptive_tokens"].tolist())
    out["adaptive_pred"] = st["pred"]
    out["adaptive_r_feat"], out["adaptive_r_words"], _ = O.adaptive_explain_wordt(asd, st, ADA["T"] - 1)
    out["block_mask"] = O.block_image(inp["heat"].mean((0, 1)), PATCHES, PATCH)
    out["bbox_share"] = O.bbox_ratio(inp["heat"], BOXES, THRESHOLDS)
    return out


def reference_outputs(inp):
    """The same cases through the original's own code (loaded by ref_shim)."""
    import argparse
    import torch.nn as nn
    with contextlib.redirect_stdout(io.StringIO()):
        ns = ref_shim.load_reference()
    out = {}
    # ---- encoder rules: add_lrp + compute_lrp (lrp_wrapper.py:37-87)
    net = ns.vgg.make_layers(CFG)
    net.load_state_dict(synth.vgg_state(101, CFG))
    net.eval()
    ns.lrp_wrapper.add_lrp(net)
    out["conv_stack_rel"] = net.compute_lrp(inp["conv_x"].clone(), target=inp["conv_target"])
    # ---- tuner weights: GridTDModel.get_lrp_weight_step (gridTDmodel.py:549-578)
    V = LW["V"]
    stop, wm = synth.stop_mask(V), synth.word_map(V)
    rev = {v: ("the" if (bool(stop[v]) and k.startswith("w")) else k) for k, v in wm.items()}
    with contextlib.redirect_stdout(io.StringIO()):
        gm = ns.gridTDmodel.GridTDModel(LW["E"], LW["H"], V, "vgg16")
    gm.load_state_dict(synth.gridtd_decoder_state(103, V, LW["H"], LW["E"]), strict=False)
    with torch.no_grad():
        out["w_ctx"], out["w_h"] = gm.get_lrp_weight_step(inp["logits"], rev, inp["h"], inp["c"])
    # ---- ExplainAdaptiveAttention (adaptiveattention.py:626-771)
    V, H, T = ADA["V"], ADA["H"], ADA["T"]
    with contextlib.redirect_stdout(io.StringIO()):
        am = ns.adaptiveattention.AdaptiveAttentionCaptioningModel(H, H, V, "vgg16")
    am.load_state_dict(synth.adaptive_decoder_state(105, V, H, H), strict=False)
    feats, toks = inp["adaptive_feats"], inp["adaptive_tokens"].tolist()

    class _Enc(nn.Module):
        encoder = nn.Identity()

        def forward(self, img):
            return feats, feats.mean((2, 3)).squeeze()

    am.img_encoder = _Enc()
    am.beam_search = lambda *a, **k: ([" ".join(f"w{t}" for t in toks[1:])], toks[1:])
    args = argparse.Namespace(embed_dim=H, hidden_dim=H, encoder="vgg16", height=224, width=224, save_path="/tmp/lrpx_ref",
                              dataset="syn", weight="")
    os.makedirs("/tmp/lrpx_ref", exist_ok=True)
    ex = ns.adaptiveattention.ExplainAdaptiveAttention(args, synth.word_map(V), model=am)
    ex.preprocess_img = lambda p: torch.zeros(1, 3, 224, 224)
    with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
        ex.get_hidden_parameters("x")
        rf_ref, rw_ref = ex.explain_caption_wordt(T - 1)
    out["adaptive_pred"] = ex.predictions
    out["adaptive_r_feat"], out["adaptive_r_words"] = rf_ref[0].reshape(512, -1).t(), rw_ref
    # ---- evaluation.py: block_image (:57-80) and the bbox share (:310-342)
    ev = ref_shim.load_reference_evaluation()

    class _Ex:
        model = nn.Identity()
        word_map = {"<start>": 0}

    exp = ev.EvaluationExperiments(_Ex())
    assert (exp.num_delete_patches, exp.patch_size) == (PATCHES, PATCH), (exp.num_delete_patches, exp.patch_size)
    heat = inp["heat"]
    with contextlib.redirect_stdout(io.StringIO()):
        out["block_mask"] = exp.block_image(torch.mean(heat, dim=(0, 1)))
    rel = exp._project_maxabs(np.mean(np.maximum(heat.numpy().copy(), 0), axis=(0, 1)))
    out["bbox_share"] = torch.tensor([[exp._calculate_overlaped_pixels(b, rel, t) for t in THRESHOLDS] for b in BOXES])
    return out


def compare(actual, expected, what):
    """Asserts every output of BARS within its bar; prints one `ok` line per output."""
    for name, (rtol, atol) in BARS.items():
        a, b = torch.as_tensor(actual[name]).detach().double(), torch.as_tensor(expected[name]).detach().double()
        assert a.shape == b.shape, f"{what} {name}: shape {tuple(a.shape)} != {tuple(b.shape)}"
        if name == "adaptive_r_feat":
            scale = float(b.abs().max())
            a, b = a / scale, b / scale
        bad = (a - b).abs() > atol + rtol * b.abs()
        assert not bool(bad.any()), (f"MISMATCH {what} {name}: {int(bad.sum())}/{bad.numel()} worst "
                                     f"{float((a - b).abs().max()):.3e}")
        print(f"ok {what} {name}: max abs diff {float((a - b).abs().max()):.3e}")


def load_fixture(path=FIXTURE):
    """-> (inputs, expected outputs, source)"""
    d = np.load(path, allow_pickle=False)
    inp = {k[3:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("in_")}
    exp = {k[4:]: torch.from_numpy(d[k]) for k in d.files if k.startswith("out_")}
    return inp, exp, str(d["source"])


def store(inp, outputs, source, path=FIXTURE):
    arrays = {"in_" + k: v.numpy() for k, v in inp.items()}
    arrays.update({"out_" + k: torch.as_tensor(outputs[k]).detach().float().numpy() for k in BARS})
    np.savez_compressed(path, source=np.array(source), **arrays)
    print(f"stored {path} (expected outputs: {source})")


def main(argv):
    live = ref_shim.reference_available()
    if not live and "--store" not in argv:
        print("original not available")
        return 77
    inp = case_inputs()
    ours = oracle_outputs(inp)
    if live:
        ref = reference_outputs(inp)
        compare(ours, ref, "oracle vs original")
        if "--store" not in argv:
            compare(load_fixture()[1], ref, "stored vs original")
    if "--store" in argv:
        store(inp, ref if live else ours, "original" if live else "oracle (lrp_oracle.py)")
    return 0


if __name__ == "__main__":
    sys.exit(main(sys.argv[1:]))
