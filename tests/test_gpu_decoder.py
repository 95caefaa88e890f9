"""GPU parity: batched decoder relevance kernels (gridTD / AoA explain_caption_wordt) vs the fixtures generated
by the reference's ExplainGridTDAttention / ExplainAOAAttention, and vs the oracle on multi-image batches."""
import pytest
import torch

import helpers
import lrp_oracle as O
import synth
from conftest import assert_close
from lrpx import decoder as D

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _ref_feat(r, C):
    """(1,C,h,w) fixture -> (P,C) pixel-major."""
    return r[0].reshape(C, -1).t()


@pytest.mark.parametrize("tc_gemm", [False, True])
@pytest.mark.parametrize("name", ["gridtd_dec_small", "gridtd_dec_512"])
def test_gridtd_vs_reference_fixture(golden, name, tc_gemm):
    """tc_gemm=True: the GEMMs run as error-compensated bf16x3 on the tensor cores (~2^-16 relative per product);
    bar for that mode: scale-relative atol 1e-4 (fp32 CUDA-core mode: 1e-5)."""
    from lrpx import ops
    g = golden(name)
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    p = synth.gridtd_decoder_state(int(g["seed"]), V, H, E)
    toks = g["tokens"].tolist()
    st = O.gridtd_explainer_forward(p, g["feats"][0], toks)
    ks = helpers.gridtd_kernel_state([st], DEV)
    W = helpers.to_dev(D.gridtd_weights(p), DEV)
    ts = g["ts"].tolist()
    req_img = torch.zeros(len(ts), dtype=torch.int32)
    req_t = torch.tensor(ts, dtype=torch.int32)
    req_word = torch.tensor([toks[t + 1] for t in ts], dtype=torch.int32)
    r_feat, r_words, raw = ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, want_raw=True, tc_gemm=tc_gemm)
    atol = 1e-4 if tc_gemm else 1e-5
    for q, t in enumerate(ts):
        ref = _ref_feat(g[f"r_feat_{t}"], 512)
        scale = ref.abs().max()
        print(f"{name} tc_gemm={tc_gemm} t={t}: max scale-relative error "
              f"{float((r_feat[q].cpu() - ref).abs().max() / scale):.3e}")
        assert_close(r_feat[q] / scale, ref / scale, rtol=1e-4, atol=atol, what=f"{name} r_feat t={t}")
        assert_close(r_words[q, :t + 1], g[f"r_words_{t}"], rtol=1e-4, atol=atol, what=f"{name} r_words t={t}")
        assert float(r_words[q, t + 1:].abs().sum()) == 0.0
        # conservation report: relevance reaching the features + words vs the explained logit
        print(f"{name} t={t}: sum r_feat={float(r_feat[q].sum()):.6g} sum r_words_raw={float(raw[q].sum()):.6g} "
              f"logit={float(st['pred'][t][toks[t + 1]]):.6g}")


def test_gridtd_batched_requests_vs_oracle():
    """Several images with ragged caption lengths, requests in arbitrary order (incl. duplicates and t=0)."""
    from lrpx import ops
    V, H, E = 120, 64, 32
    p = synth.gridtd_decoder_state(7, V, H, E, C=64, n_pixel=16)
    states, toks = [], []
    for b, T in enumerate([5, 3, 1]):
        f = torch.randn(64, 4, 4, generator=torch.Generator().manual_seed(100 + b)).clamp(min=0)
        tk = synth.tokens(200 + b, T, V)
        toks.append(tk)
        states.append(O.gridtd_explainer_forward(p, f, tk))
    ks = helpers.gridtd_kernel_state(states, DEV)
    W = helpers.to_dev(D.gridtd_weights(p), DEV)
    reqs = [(0, 4), (1, 0), (2, 0), (0, 0), (1, 2), (0, 4), (0, 2)]
    req_img = torch.tensor([r[0] for r in reqs], dtype=torch.int32)
    req_t = torch.tensor([r[1] for r in reqs], dtype=torch.int32)
    req_word = torch.tensor([toks[b][t + 1] for b, t in reqs], dtype=torch.int32)
    r_feat, r_words = ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word)
    for q, (b, t) in enumerate(reqs):
        rf, rw, _ = O.gridtd_explain_wordt({k: v.double() for k, v in p.items()},
                                           {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v)
                                            for k, v in states[b].items()}, t)
        scale = rf.abs().max()
        assert_close(r_feat[q] / scale, rf / scale, rtol=1e-3, atol=2e-5, what=f"req {q} r_feat")
        assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=2e-5, what=f"req {q} r_words")
    # zero requests is a no-op
    e = torch.zeros(0, dtype=torch.int32)
    rf0, rw0 = ops.gridtd_decoder_lrp(ks, W, e, e, e)
    assert rf0.shape[0] == 0 and rw0.shape[0] == 0


@pytest.mark.parametrize("tc_gemm", [False, True])
@pytest.mark.parametrize("name", ["aoa_dec_512", "aoa_dec_bu"])
def test_aoa_vs_reference_fixture(golden, name, tc_gemm):
    from lrpx import ops
    g = golden(name)
    V, H, E, C = int(g["V"]), int(g["H"]), int(g["E"]), int(g["C"])
    p = synth.aoa_decoder_state(int(g["seed"]), V, H, E, C)
    toks = g["tokens"].tolist()
    st = O.aoa_explainer_forward(p, g["feats"][0], toks, 8)
    ks = helpers.aoa_kernel_state([st], DEV)
    W = helpers.to_dev(D.aoa_weights(p), DEV)
    cases = g["cases"].tolist()
    req_img = torch.zeros(len(cases), dtype=torch.int32)
    req_t = torch.tensor([c[0] for c in cases], dtype=torch.int32)
    req_head = torch.tensor([c[1] for c in cases], dtype=torch.int32)
    req_word = torch.tensor([toks[c[0] + 1] for c in cases], dtype=torch.int32)
    r_feat, r_words = ops.aoa_decoder_lrp(ks, W, 8, req_img, req_t, req_word, req_head, tc_gemm=tc_gemm)
    atol = 1e-4 if tc_gemm else 1e-5
    for q, (t, hd) in enumerate(cases):
        ref = _ref_feat(g[f"r_feat_{t}_{hd}"], C)
        scale = ref.abs().max()
        print(f"{name} tc_gemm={tc_gemm} ({t},{hd}): max scale-relative error "
              f"{float((r_feat[q].cpu() - ref).abs().max() / scale):.3e}")
        assert_close(r_feat[q] / scale, ref / scale, rtol=1e-4, atol=atol, what=f"{name} r_feat {t},{hd}")
        assert_close(r_words[q, :t + 1], g[f"r_words_{t}_{hd}"], rtol=1e-4, atol=atol, what=f"{name} r_words {t},{hd}")


@pytest.mark.parametrize("tc_gemm", [False, True])
@pytest.mark.parametrize("name", ["adaptive_dec_small", "adaptive_dec_512"])
def test_adaptive_vs_reference_fixture(golden, name, tc_gemm):
    """SURVEY §8 f2: lrpx_adaptive_decoder_lrp_f32 vs ExplainAdaptiveAttention.explain_caption_wordt run by the
    reference (adaptiveattention.py:679-771).  Same bars as the gridTD kernel."""
    from lrpx import ops
    g = golden(name)
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    p = synth.adaptive_decoder_state(int(g["seed"]), V, H, E)
    toks = g["tokens"].tolist()
    st = O.adaptive_explainer_forward(p, g["feats"][0], toks)
    ks = helpers.adaptive_kernel_state([st], DEV)
    W = helpers.to_dev(D.adaptive_weights(p), DEV)
    ts = g["ts"].tolist()
    req_img = torch.zeros(len(ts), dtype=torch.int32)
    req_t = torch.tensor(ts, dtype=torch.int32)
    req_word = torch.tensor([toks[t + 1] for t in ts], dtype=torch.int32)
    r_feat, r_words, raw = ops.adaptive_decoder_lrp(ks, W, req_img, req_t, req_word, want_raw=True, tc_gemm=tc_gemm)
    atol = 1e-4 if tc_gemm else 1e-5
    for q, t in enumerate(ts):
        ref = _ref_feat(g[f"r_feat_{t}"], 512)
        scale = ref.abs().max()
        print(f"{name} tc_gemm={tc_gemm} t={t}: max scale-relative error "
              f"{float((r_feat[q].cpu() - ref).abs().max() / scale):.3e}")
        assert_close(r_feat[q] / scale, ref / scale, rtol=1e-4, atol=atol, what=f"{name} r_feat t={t}")
        assert_close(r_words[q, :t + 1], g[f"r_words_{t}"], rtol=1e-4, atol=atol, what=f"{name} r_words t={t}")
        assert float(r_words[q, t + 1:].abs().sum()) == 0.0
        print(f"{name} t={t}: sum r_feat={float(r_feat[q].sum()):.6g} sum r_words_raw={float(raw[q].sum()):.6g} "
              f"logit={float(st['pred'][t][toks[t + 1]]):.6g}")


def test_adaptive_batched_requests_vs_oracle():
    """Several images with ragged caption lengths, requests in arbitrary order (duplicates, t=0), empty batch."""
    from lrpx import ops
    V, H, E = 120, 64, 64
    p = synth.adaptive_decoder_state(8, V, H, E, C=96, n_pixel=16)
    states, toks = [], []
    for b, T in enumerate([5, 3, 1]):
        f = torch.randn(96, 4, 4, generator=torch.Generator().manual_seed(300 + b)).clamp(min=0)
        tk = synth.tokens(400 + b, T, V)
        toks.append(tk)
        states.append(O.adaptive_explainer_forward(p, f, tk))
    ks = helpers.adaptive_kernel_state(states, DEV)
    W = helpers.to_dev(D.adaptive_weights(p), DEV)
    reqs = [(0, 4), (1, 0), (2, 0), (0, 0), (1, 2), (0, 4), (0, 2)]
    req_img = torch.tensor([r[0] for r in reqs], dtype=torch.int32)
    req_t = torch.tensor([r[1] for r in reqs], dtype=torch.int32)
    req_word = torch.tensor([toks[b][t + 1] for b, t in reqs], dtype=torch.int32)
    r_feat, r_words = ops.adaptive_decoder_lrp(ks, W, req_img, req_t, req_word)
    pd = {k: v.double() for k, v in p.items()}
    for q, (b, t) in enumerate(reqs):
        rf, rw, _ = O.adaptive_explain_wordt(pd, {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v)
                                                  for k, v in states[b].items()}, t)
        scale = rf.abs().max()
        assert_close(r_feat[q] / scale, rf / scale, rtol=1e-3, atol=2e-5, what=f"req {q} r_feat")
        assert_close(r_words[q, :t + 1], rw, rtol=1e-3, atol=2e-5, what=f"req {q} r_words")
    e = torch.zeros(0, dtype=torch.int32)
    rf0, rw0 = ops.adaptive_decoder_lrp(ks, W, e, e, e)
    assert rf0.shape[0] == 0 and rw0.shape[0] == 0


def test_gridtd_persistent_workspace_keeps_prepared_weights(golden):
    """ops.gridtd_decoder_lrp(..., ws_cache=dict): the workspace of a shape and weights is kept and later calls on it
    skip the weight conversion (LRPX_DEC_W3_READY) — bit-identical results, one entry per argument shape and weights
    (other weights, or the same ones updated in place, get their own entry: test_gpu_weight_updates.py)."""
    from lrpx import ops
    g = golden("gridtd_dec_512")
    V, H, E = int(g["V"]), int(g["H"]), int(g["E"])
    p = synth.gridtd_decoder_state(int(g["seed"]), V, H, E)
    toks = g["tokens"].tolist()
    st = O.gridtd_explainer_forward(p, g["feats"][0], toks)
    ks = helpers.gridtd_kernel_state([st], DEV)
    W = helpers.to_dev(D.gridtd_weights(p), DEV)
    ts = g["ts"].tolist()
    req_img = torch.zeros(len(ts), dtype=torch.int32)
    req_t = torch.tensor(ts, dtype=torch.int32)
    req_word = torch.tensor([toks[t + 1] for t in ts], dtype=torch.int32)
    ref = ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, tc_gemm=True)
    cache = {}
    first = ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, tc_gemm=True, ws_cache=cache)
    assert len(cache) == 1
    ws = next(iter(cache.values()))
    again = ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, tc_gemm=True, ws_cache=cache)       # READY path
    assert len(cache) == 1 and next(iter(cache.values())) is ws
    for a, b, c in zip(ref, first, again):
        assert torch.equal(a, b) and torch.equal(a, c)
    # another request count is another shape: its own workspace, same results for the shared requests
    sub = ops.gridtd_decoder_lrp(ks, W, req_img[:1], req_t[:1], req_word[:1], tc_gemm=True, ws_cache=cache)
    sub2 = ops.gridtd_decoder_lrp(ks, W, req_img[:1], req_t[:1], req_word[:1], tc_gemm=True, ws_cache=cache)
    assert len(cache) == 2
    assert torch.equal(sub[0], ref[0][:1]) and torch.equal(sub2[0], ref[0][:1])
    # fp32 CUDA-core GEMMs never cache
    ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, tc_gemm=False, ws_cache=cache)
    assert len(cache) == 2
