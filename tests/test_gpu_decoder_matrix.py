"""Parity matrix of the six batched decoder entry points (gridTD / AoA / adaptive, LRP relevance and gradient) against
the float64 oracle, across the routes their GEMMs take.

Each GEMM of a decoder picks its own route: the error-compensated bf16x3 tensor-core GEMM when ``tc_gemm`` is set and
``tc_shape_ok(N, K)`` holds, the fp32 CUDA-core SGEMM otherwise.  The route also decides which workspace slot receives
the split operand (``a3``, or ``a3u`` when the step kernels write the split themselves).  SHAPES runs every GEMM of
every decoder on both routes and the fused split both on and off; ``test_route_table_covers_both_routes`` (no GPU)
keeps that list honest, and ``test_workspace_holds_weight_copies_and_split_operands`` (no GPU) checks the workspace
sizes against the same GEMM table.  Further cases: odd hidden widths and pixel counts, the long-caption fallback of the gridTD
relevance attention, workspace sizing with E > 4H, request counts beyond a grid's y limit (65 535), a second device.

Bars: scale-relative atol 1e-5 on the CUDA-core route, 1e-4 on the tensor-core route (bf16x3 keeps ~2^-16 relative per
product), rtol 1e-4 on both."""
import functools

import pytest
import torch

import helpers
import lrp_oracle as O
import synth
from conftest import assert_close
from lrpx import decoder as D

DEV = "cuda"


# ------------------------------------------------------------------------------------------------ route table (CPU)
def tc_shape_ok(N, K):
    """``tc_shape_ok`` of csrc/dec_gemm.cuh — the shapes the tensor-core GEMM takes (N output columns, K reduction
    length)."""
    return K % 64 == 0 and N % 32 == 0 and (N <= 256 or N % 256 == 0)


def gemm_table(kind, H, E, C, Q=1, P=1):
    """(weight, N, K, rows) of every GEMM the entry point runs for Q requests of P pixels (csrc/decoder.cu,
    csrc/decoder_grad.cu)."""
    QP = Q * P
    return {
        "gridtd_lrp": [("W_g2", 3 * H, H, Q), ("W_g1", 2 * H + 2 * E, H, Q), ("W_glob", C, E, Q), ("W_proj", C, H, QP)],
        "aoa_lrp": [("W_aoa", H, H, Q), ("W_g", E + 2 * H, H, Q), ("W_v", H, H, QP), ("W_proj", C, H, QP)],
        "adaptive_lrp": [("W_g", 2 * E + H, H, Q), ("W_glob", C, E, Q), ("W_proj", C, H, QP)],
        "gridtd_grad": [("W2", 3 * H, 4 * H, Q), ("W1", H + 2 * E, 4 * H, Q), ("W_glob", C, E, Q), ("W_proj", C, H, QP)],
        "aoa_grad": [("W_aoa", H, H, Q), ("W_gate", H, H, Q), ("W_g", E + 2 * H, 4 * H, Q), ("W_v", H, H, QP),
                     ("W_proj", C, H, QP)],
        "adaptive_grad": [("W_g", 2 * E + H, 4 * H, Q), ("W_glob", C, E, Q), ("W_proj", C, H, Q)],
    }[kind]


# step GEMMs whose operand the step kernels split themselves when all of them run on the tensor cores
FUSED = {"gridtd_lrp": ("W_g2", "W_g1"), "gridtd_grad": ("W2", "W1"), "adaptive_lrp": ("W_g",)}
KINDS = ["gridtd_lrp", "aoa_lrp", "adaptive_lrp", "gridtd_grad", "gridtd_guided", "aoa_grad", "adaptive_grad"]
# (H, E, C)
SHAPES = [(64, 64, 256), (64, 48, 96), (64, 40, 64), (96, 64, 512), (32, 32, 64), (128, 64, 256)]


def _gemm_kind(kind):
    return "gridtd_grad" if kind == "gridtd_guided" else kind


def test_route_table_covers_both_routes():
    """With tc_gemm, every GEMM of every decoder meets the tensor-core route at some shape of SHAPES and the CUDA-core
    route at another, and the fused operand split runs on and off."""
    for kind in dict.fromkeys(map(_gemm_kind, KINDS)):
        seen = {}
        fused_states = set()
        for H, E, C in SHAPES:
            routes = {name: tc_shape_ok(N, K) for name, N, K, _ in gemm_table(kind, H, E, C)}
            for name, tc in routes.items():
                seen.setdefault(name, set()).add(tc)
            if kind in FUSED:
                fused_states.add(all(routes[n] for n in FUSED[kind]))
        for name, routes in seen.items():
            assert routes == {False, True}, f"{kind} {name}: only the {'tensor' if True in routes else 'CUDA'}-core route"
        if kind in FUSED:
            assert fused_states == {False, True}, f"{kind}: fused split only {fused_states}"


def test_route_table_edge_cases():
    """The shapes the workspace and wide-grid tests rely on take the routes their docstrings name."""
    # adaptive gradient at (32, 192, 512): only W_glob on the tensor cores, and it splits Q x E with E > 4H
    routes = {n: tc_shape_ok(N, K) for n, N, K, _ in gemm_table("adaptive_grad", 32, 192, 512)}
    assert routes == {"W_g": False, "W_glob": True, "W_proj": False}
    # (64, 64, 64): every GEMM of every decoder on the tensor cores
    for kind in dict.fromkeys(map(_gemm_kind, KINDS)):
        assert all(tc_shape_ok(N, K) for _, N, K, _ in gemm_table(kind, 64, 64, 64)), kind


def test_workspace_holds_weight_copies_and_split_operands():
    """With tc_gemm the workspace grows by at least the prepared copy of every weight (N x 3K bf16, stored
    [hi | hi | lo]) plus the largest split operand (rows x 2K bf16, stored [hi | lo]) of the decoder's GEMMs.  A slot
    sized by a smaller formula lets that split overwrite the slot next to it.  Host calls: no GPU needed."""
    import ctypes
    from lrpx import _lib
    lib = _lib.lib()
    entry = {"gridtd_lrp": (_lib.GridTDArgs, lib.lrpx_gridtd_decoder_workspace_bytes),
             "aoa_lrp": (_lib.AoaArgs, lib.lrpx_aoa_decoder_workspace_bytes),
             "adaptive_lrp": (_lib.AdaptiveArgs, lib.lrpx_adaptive_decoder_workspace_bytes),
             "gridtd_grad": (_lib.GridTDGradArgs, lib.lrpx_gridtd_decoder_grad_workspace_bytes),
             "aoa_grad": (_lib.AoaGradArgs, lib.lrpx_aoa_decoder_grad_workspace_bytes),
             "adaptive_grad": (_lib.AdaptiveGradArgs, lib.lrpx_adaptive_decoder_grad_workspace_bytes)}
    Q, P = 16, 7
    for kind in dict.fromkeys(map(_gemm_kind, KINDS)):
        args_cls, ws_bytes = entry[kind]
        for H, E, C in SHAPES + [(32, 192, 512), (36, 64, 64), (30, 64, 64)]:
            dims = dict(B=3, T=5, H=H, E=E, P=P, C=C, V=40, Q=Q)
            if kind.startswith("aoa"):
                dims["num_head"] = heads_for(H)
            size = lambda flags: ws_bytes(ctypes.byref(args_cls(**dims, flags=flags)))
            table = gemm_table(kind, H, E, C, Q, P)
            need = sum(2 * N * 3 * K for _, N, K, _ in table) + 2 * max(rows * 2 * K for _, _, K, rows in table)
            assert size(1) - size(0) >= need, f"{kind} (H, E, C) = {(H, E, C)}"


def heads_for(H):
    return next(n for n in (8, 6, 4) if H % n == 0)


# ------------------------------------------------------------------------------------------------ state and oracle
def _family(kind):
    return kind.split("_")[0]


def _is_grad(kind):
    return not kind.endswith("_lrp")


@functools.lru_cache(maxsize=None)
def _case(family, gradient, H, E, C, P, Ts, seed=0):
    """Seeded decoder weights and one oracle explainer forward (float32) per image, captions of lengths Ts."""
    V = 40
    if family == "gridtd":
        p = synth.gridtd_decoder_state(seed + 11, V, H, E, C=C, n_pixel=P)
    elif family == "aoa":
        p = synth.aoa_decoder_state(seed + 12, V, H, E, C=C)
    else:
        p = synth.adaptive_decoder_state(seed + 13, V, H, E, C=C, n_pixel=P)
    nh = heads_for(H)
    states, toks = [], []
    for b, T in enumerate(Ts):
        f = torch.randn(C, P, 1, generator=torch.Generator().manual_seed(seed + 100 + b)).clamp(min=0)
        tk = synth.tokens(seed + 200 + b, T, V)
        toks.append(tk)
        if family == "gridtd":
            states.append(O.gridtd_explainer_forward(p, f, tk, gradient=gradient))
        elif family == "aoa":
            states.append(O.aoa_explainer_forward(p, f, tk, nh, gradient=gradient))
        else:
            states.append(O.adaptive_explainer_forward(p, f, tk))
    return p, states, toks, nh


def adaptive_grad_kernel_state(oracle_states, device):
    """oracle.adaptive_explainer_forward dicts -> stacked state of lrpx_adaptive_grad_args"""
    step = D.ADAPTIVE_STEP_KEYS + ["o", "sg"]
    keys = D.ADAPTIVE_IMAGE_KEYS + step + D.ADAPTIVE_STEP1_KEYS
    conv = [{k: st[helpers._GRID_RENAME.get(k, k)] for k in keys} for st in oracle_states]
    return D.stack_states(conv, D.ADAPTIVE_IMAGE_KEYS, step, D.ADAPTIVE_STEP1_KEYS, device)


@functools.lru_cache(maxsize=None)
def _kernel_inputs(kind, H, E, C, P, Ts, device=DEV):
    """(state, weights) of the entry point on ``device``."""
    from models._gradient import aoa_grad_weights, gridtd_grad_weights
    from models.adaptiveattention import adaptive_grad_weights
    kind = _gemm_kind(kind)
    p, states, _, _ = _case(_family(kind), _is_grad(kind), H, E, C, P, Ts)
    state_fn, weight_fn = {
        "gridtd_lrp": (helpers.gridtd_kernel_state, D.gridtd_weights),
        "aoa_lrp": (helpers.aoa_kernel_state, D.aoa_weights),
        "adaptive_lrp": (helpers.adaptive_kernel_state, D.adaptive_weights),
        "gridtd_grad": (helpers.gridtd_grad_kernel_state, gridtd_grad_weights),
        "aoa_grad": (helpers.aoa_grad_kernel_state, aoa_grad_weights),
        "adaptive_grad": (adaptive_grad_kernel_state, adaptive_grad_weights),
    }[kind]
    return state_fn(states, device), helpers.to_dev(weight_fn(p), device)


def run_kernel(kind, H, E, C, P, Ts, reqs, tc_gemm, want_raw=False, device=DEV):
    """reqs: (image, t, head) -> the entry point's outputs for those requests (head is ignored outside AoA)."""
    from lrpx import ops
    ks, W = _kernel_inputs(kind, H, E, C, P, Ts, device)
    _, _, toks, nh = _case(_family(_gemm_kind(kind)), _is_grad(kind), H, E, C, P, Ts)
    i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=device)
    req_img, req_t = i32([b for b, _, _ in reqs]), i32([t for _, t, _ in reqs])
    req_word, req_head = i32([toks[b][t + 1] for b, t, _ in reqs]), i32([h for _, _, h in reqs])
    kw = dict(want_raw=want_raw, tc_gemm=tc_gemm)
    if kind == "gridtd_lrp":
        return ops.gridtd_decoder_lrp(ks, W, req_img, req_t, req_word, **kw)
    if kind == "aoa_lrp":
        return ops.aoa_decoder_lrp(ks, W, nh, req_img, req_t, req_word, req_head, **kw)
    if kind == "adaptive_lrp":
        return ops.adaptive_decoder_lrp(ks, W, req_img, req_t, req_word, **kw)
    if kind in ("gridtd_grad", "gridtd_guided"):
        return ops.gridtd_decoder_grad(ks, W, req_img, req_t, req_word, guided=kind == "gridtd_guided", **kw)
    if kind == "aoa_grad":
        return ops.aoa_decoder_grad(ks, W, nh, req_img, req_t, req_word, req_head, **kw)
    return ops.adaptive_decoder_grad(ks, W, req_img, req_t, req_word, **kw)


def _dbl(d):
    return {k: (v.double() if torch.is_tensor(v) and v.is_floating_point() else v) for k, v in d.items()}


@functools.lru_cache(maxsize=None)
def oracle(kind, H, E, C, P, Ts, b, t, head):
    """float64 oracle of one request -> (r_feat (P, C), r_words (t+1,), raw r_words (t+1,) or None, scale of the raw
    r_words: max over words of the sum of |r_emb|, the terms each raw value sums)."""
    p, states, _, _ = _case(_family(_gemm_kind(kind)), _is_grad(kind), H, E, C, P, Ts)
    pd, sd = _dbl(p), _dbl(states[b])
    if kind == "gridtd_lrp":
        rf, rw, ex = O.gridtd_explain_wordt(pd, sd, t)
    elif kind == "aoa_lrp":
        rf, rw, ex = O.aoa_explain_wordt(pd, sd, t, head)
    elif kind == "adaptive_lrp":
        rf, rw, ex = O.adaptive_explain_wordt(pd, sd, t)
    elif kind in ("gridtd_grad", "gridtd_guided"):
        (rf, rw), ex = O.gridtd_gradient_wordt(pd, sd, t, guided=kind == "gridtd_guided"), None
    elif kind == "aoa_grad":
        (rf, rw), ex = O.aoa_gradient_wordt(pd, sd, t, head), None
    else:
        (rf, rw), ex = O.adaptive_gradient_wordt(pd, sd, t), None
    if ex is None:
        return rf, rw, None, None
    return rf, rw, ex["r_emb"].sum(-1), float(ex["r_emb"].abs().sum(-1).max())


def bar(tc_gemm):
    return 1e-4 if tc_gemm else 1e-5


def check_requests(kind, H, E, C, P, Ts, reqs, out, tc_gemm, qs=None, what=""):
    """Every request q in ``qs`` (default: all) against the oracle; r_words exactly zero past t; the raw word relevance
    (when ``out`` carries it) against the oracle's (LRP) or as the pre-normalisation form of r_words (gradient)."""
    r_feat, r_words = out[0], out[1]
    raw = out[2] if len(out) > 2 else None
    atol = bar(tc_gemm)
    for q in (range(len(reqs)) if qs is None else qs):
        b, t, hd = reqs[q]
        rf, rw, rraw, raw_scale = oracle(kind, H, E, C, P, Ts, b, t, hd)
        tag = f"{what} {kind} tc_gemm={tc_gemm} request {q} (image {b}, t={t}, head {hd})"
        scale = float(rf.abs().max())
        assert scale > 0, tag
        assert_close(r_feat[q] / scale, rf / scale, rtol=1e-4, atol=atol, what=f"{tag} r_feat")
        assert_close(r_words[q, :t + 1], rw, rtol=1e-4, atol=atol, what=f"{tag} r_words")
        assert float(r_words[q, t + 1:].abs().sum()) == 0.0, f"{tag}: r_words past t"
        if raw is not None:
            assert float(raw[q, t + 1:].abs().sum()) == 0.0, f"{tag}: raw r_words past t"
            rq = raw[q, :t + 1]
            if rraw is not None:        # a word's raw value is a sum of E terms of both signs: scaled by their magnitude
                assert_close(rq / raw_scale, rraw / raw_scale, rtol=1e-4, atol=atol, what=f"{tag} raw r_words")
            else:
                assert_close(rq / rq.abs().max(), rw, rtol=1e-4, atol=atol, what=f"{tag} raw r_words")


# several images with ragged captions (incl. T_b = 1); requests in arbitrary order with duplicates, t = 0 and
# t = T_b - 1; on AoA request q follows head q % num_head, so every head is explained
TS = (5, 3, 1)
REQS = [(0, 4), (1, 0), (2, 0), (0, 0), (1, 2), (0, 4), (0, 2), (1, 1), (0, 3)]


def _reqs(kind, H, base=REQS):
    nh = heads_for(H) if _family(kind) == "aoa" else 1
    return [(b, t, q % nh) for q, (b, t) in enumerate(base)]


@pytest.mark.gpu
@pytest.mark.parametrize("tc_gemm", [False, True])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "H%d-E%d-C%d" % s)
@pytest.mark.parametrize("kind", KINDS)
def test_decoder_matrix_vs_oracle(kind, shape, tc_gemm):
    H, E, C = shape
    P = 16
    reqs = _reqs(kind, H)
    if _family(kind) == "aoa":
        assert {h for _, _, h in reqs} == set(range(heads_for(H)))
    out = run_kernel(kind, H, E, C, P, TS, reqs, tc_gemm, want_raw=True)
    check_requests(kind, H, E, C, P, TS, reqs, out, tc_gemm)
    # the same requests without the raw output: identical results
    plain = run_kernel(kind, H, E, C, P, TS, reqs, tc_gemm)
    assert torch.equal(plain[0], out[0]) and torch.equal(plain[1], out[1])


@pytest.mark.gpu
@pytest.mark.parametrize("kind", KINDS)
def test_decoder_zero_requests_is_a_no_op(kind):
    H, E, C = SHAPES[0]
    for tc_gemm in (False, True):
        out = run_kernel(kind, H, E, C, 16, TS, [], tc_gemm, want_raw=True)
        assert out[0].shape == (0, 16, C) and out[1].shape == (0, max(TS)) and out[2].shape == (0, max(TS))


@pytest.mark.gpu
@pytest.mark.parametrize("tc_gemm", [False, True])
@pytest.mark.parametrize("P", [16, 7, 1])
@pytest.mark.parametrize("H", [36, 30])
@pytest.mark.parametrize("kind", KINDS)
def test_decoder_odd_widths_and_pixel_counts(kind, H, P, tc_gemm):
    """H = 36 (a multiple of 4, not of 8) and H = 30 (not a multiple of 4); P = 16 (the attention kernels' vector path),
    7 (a tail) and 1.  Only the gridTD gradient entry point requires H % 4 == 0 and refuses H = 30."""
    from lrpx import _lib
    E, C = 64, 64
    reqs = _reqs(kind, H)
    if H % 4 and kind in ("gridtd_grad", "gridtd_guided"):
        with pytest.raises(_lib.LrpxError, match="multiple of 4"):
            run_kernel(kind, H, E, C, P, TS, reqs, tc_gemm)
        return
    out = run_kernel(kind, H, E, C, P, TS, reqs, tc_gemm, want_raw=True)
    check_requests(kind, H, E, C, P, TS, reqs, out, tc_gemm)


@pytest.mark.gpu
@pytest.mark.parametrize("tc_gemm", [False, True])
def test_gridtd_lrp_long_caption_wide_state_vs_oracle(tc_gemm):
    """T x (P + H) beyond the shared memory of the row-wise attention kernel (45 steps, H = 1152, P = 16): the
    per-(pixel, request) fallback grid_attn_kernel runs; same results as the oracle."""
    H, E, C, P, T = 1152, 64, 64, 16, 45
    assert T * (P + H) * 4 > 160 * 1024
    reqs = [(0, T - 1, 0), (0, 7, 0), (0, 0, 0)]
    out = run_kernel("gridtd_lrp", H, E, C, P, (T,), reqs, tc_gemm, want_raw=True)
    check_requests("gridtd_lrp", H, E, C, P, (T,), reqs, out, tc_gemm)


@pytest.mark.gpu
def test_adaptive_grad_workspace_with_embed_wider_than_4h():
    """Adaptive gradient at (H, E, C) = (32, 192, 512), tensor-core GEMMs, P = 4: only the W_glob GEMM runs on the
    tensor cores and it splits d_glob (Q x E, E = 6H) into the operand slot.  That slot must hold Q x 2E bf16, not
    only Q x 2 x 4H: 2048 requests (16 distinct (image, t) pairs, each 128 times) against the oracle."""
    H, E, C, P, Ts = 32, 192, 512, 4, (4, 4, 4, 4)
    pairs = [(b, t, 0) for b in range(4) for t in range(4)]
    reqs = pairs * 128
    out = run_kernel("adaptive_grad", H, E, C, P, Ts, reqs, True)
    check_requests("adaptive_grad", H, E, C, P, Ts, reqs, out, True, qs=range(len(pairs)))
    n = len(pairs)
    for k in range(2):          # every repetition equals the first
        assert torch.equal(out[k].view(128, n, *out[k].shape[1:]), out[k][:n].unsqueeze(0).expand(128, *out[k][:n].shape))


@pytest.mark.gpu
@pytest.mark.parametrize("tc_gemm", [False, True])
@pytest.mark.parametrize("kind", KINDS)
def test_decoder_request_count_above_grid_y_limit(kind, tc_gemm):
    """Q = 70 000 requests (beyond the 65 535 blocks of a grid's y dimension) over 4 images, T = 3, P = 64: Q * P / 64
    row tiles exceed it too on the CUDA-core route.  The result equals the same requests computed in chunks of 4096
    bit for bit (a request's arithmetic does not depend on Q), and a sample matches the oracle."""
    H = E = C = 64
    P, Ts, Q = 64, (3, 3, 3, 3), 70000
    nh = heads_for(H) if _family(kind) == "aoa" else 1
    reqs = [(q % 4, (q // 4) % 3, (q // 12) % nh) for q in range(Q)]
    full = run_kernel(kind, H, E, C, P, Ts, reqs, tc_gemm)
    for q0 in range(0, Q, 4096):
        part = run_kernel(kind, H, E, C, P, Ts, reqs[q0:q0 + 4096], tc_gemm)
        for k in range(2):
            assert torch.equal(full[k][q0:q0 + 4096], part[k]), f"{kind} chunk at {q0}, output {k}"
    check_requests(kind, H, E, C, P, Ts, reqs, full, tc_gemm, qs=[0, 5, 13, 4097, Q - 1], what="Q=70000")


@pytest.mark.gpu
@pytest.mark.skipif(not torch.cuda.is_available() or torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_decoders_and_explainer_forward_on_a_second_device(tmp_path):
    """The kernels above 48 KB of dynamic shared memory (the gridTD relevance attention, the gridTD gradient attention,
    the explainer forward's LSTM step) run on cuda:0 and then on cuda:1 in the same process; both match the oracle."""
    import argparse
    from models import gridTDmodel as G
    H = E = C = 512
    P, Ts = 196, (19,)
    reqs = [(0, 18, 0), (0, 3, 0)]
    args = argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                              save_path=str(tmp_path), dataset="syn", weight="")
    V = 40
    for d in range(2):
        dev = f"cuda:{d}"
        with torch.cuda.device(d):
            for kind in ("gridtd_lrp", "gridtd_grad"):
                for tc_gemm in (False, True):
                    out = run_kernel(kind, H, E, C, P, Ts, reqs, tc_gemm, device=dev)
                    assert out[0].device == torch.device(dev)
                    check_requests(kind, H, E, C, P, Ts, reqs, out, tc_gemm, what=dev)
            model = G.GridTDModel(E, H, V, "vgg16")
            model.load_state_dict(synth.gridtd_decoder_state(5, V, H, E, C=C, n_pixel=P), strict=False)
            model.to(dev).eval()
            ex = G.ExplainGridTDAttention(args, synth.word_map(V), model=model, precision="fp32")
            feat = torch.randn(2, P, C, generator=torch.Generator().manual_seed(6)).clamp(min=0).to(dev)
            toks = torch.tensor([synth.tokens(7, 6, V), synth.tokens(8, 6, V)], device=dev)
            st = ex.explainer_forward(feat, toks)
            ref = helpers.gridtd_explainer_forward_ops(model, feat, toks)
            assert_close(st["pred"], ref["pred"], rtol=1e-4, atol=2e-5, what=f"{dev} explainer forward predictions")
