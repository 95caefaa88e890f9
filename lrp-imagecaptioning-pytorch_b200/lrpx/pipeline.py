"""Batched explanation pipeline: all (image, word) requests of a batch of images in one pass.

This is the throughput-oriented entry point above the reference-shaped explainers: what
``ExplainGridTDAttention.explain_caption`` does for one image (gridTDmodel.py:1141-1156: forward, then per
word decoder relevance + encoder relevance) is done here for B images x T words at once:

  encoder forward + gains (tcgen05)  ->  explainer teacher-forced forward  ->  decoder relevance kernels for
  all B*T requests  ->  encoder relevance chain (tcgen05)  ->  heat-maps (B*T,3,H,W) + r_words (B*T,T)

Optionally the whole pass is captured once into a CUDA graph (fixed B and caption length) and replayed, which
removes the launch latency of the ~2.7k small kernels of the decoder phases.  ``explain_images`` first captions the
images with the device beam search on the features of the same encoder pass.
"""
from dataclasses import dataclass

import torch

from . import _graph, ops


@dataclass
class ImageExplanation:
    """``BatchExplainer.explain_images`` for B images: Q = sum(words_per_image) requests over captions of at most T
    words."""
    captions: list            # B token lists without <start>: explain_caption's beam_caption_encode[1:]
    tokens: torch.Tensor      # (B, T+1) long: <start>, the caption, 0-padding
    words_per_image: tuple    # the B caption lengths
    req_img: torch.Tensor     # (Q,) int32: request q explains word req_t[q] + 1 of image req_img[q], image-major
    req_t: torch.Tensor       # (Q,) int32
    heat: torch.Tensor        # the Q heat-maps in the ``deliver`` format
    r_words: torch.Tensor     # (Q, T) relevance of the preceding words
    pred: torch.Tensor        # (B, T, V) logits of the explainer forward (AblationExperiments.image_ablation's pred)


class BatchExplainer:
    def __init__(self, explainer, chunk=128, use_graph=False, tc_gemm=None, head_idx=0, deliver="full"):
        """explainer: models.gridTDmodel.ExplainGridTDAttention, models.aoamodel.ExplainAOAAttention or
        models.adaptiveattention.ExplainAdaptiveAttention on a VGG encoder with precision 'fp32' (fp32-accurate chain),
        'bf16' or 'mixed', or on a Bottleneck-ResNet encoder with precision 'bf16' or 'mixed'; or one of their
        gradient-family twins (models/_gradient.py: gradient, guided backpropagation, Grad-CAM, Guided Grad-CAM; on a
        ResNet in 'bf16' / 'mixed' only Grad-CAM).  ``head_idx``: the attention head an AoA explanation follows
        (aoamodel.py:1165, ``explain_caption(img, head_idx)``); ``deliver``: format of the heat-maps
        (TcVggEngine.heat_shape): 'full' = fp32 (Q,3,H,W) like the reference, 'channel_mean' = fp32 (Q,H,W), 'fp16';
        ``tc_gemm``: decoder GEMMs as bf16x3 on tensor cores (default: with precision 'bf16') or on fp32 CUDA cores.
        Grad-CAM classes explain with their (Q, P) maps of the encoder output (what explain_cnn returns per word; the
        encoder chain does not run), so they take deliver='full' only.  Guided Grad-CAM runs the guided chain with the
        expanded Grad-CAM map applied in its last layer's epilogue, in every delivery format."""
        if not getattr(explainer, "uses_tc", False):
            raise ValueError("BatchExplainer drives the tensor-core chain: it needs a VGG-style encoder with "
                             "precision 'fp32', 'bf16' or 'mixed', or a Bottleneck ResNet with 'bf16' or 'mixed'")
        self.ex = explainer
        # gradient-family explainers (models/_gradient.py): same pipeline, the decoder-gradient kernels and the chain's
        # 'gradient' / 'guided' rule instead of the relevance ones; CAM = 'cam' (Grad-CAM) | 'guided' (Guided Grad-CAM)
        self.is_gradient = explainer.GRADIENT
        self.cam = explainer.CAM if self.is_gradient else None
        if self.cam == "cam" and deliver != "full":
            raise ValueError("Grad-CAM explains with (Q, P) maps of the encoder output: they have no channels to reduce "
                             "or store in another format, use deliver='full'")
        self._cam_px = {}         # Grad-CAM: feature-map pixels P by image size (H, W)
        self.eng = self.W = None
        self._dec_ws = {}         # persistent decoder workspaces holding the prepared copies of self.W (ops._decoder_workspace)
        self._graphs = {}
        self._sync_weights()
        self.chunk = chunk
        self.use_graph = use_graph
        # decoder GEMMs as bf16x3 on the tensor cores in both chain modes (measured 1e-5 of max off the fp32 CUDA-core
        # GEMMs, below the chain's own 2e-4 in the fp32-accurate mode); tc_gemm=False forces the CUDA-core GEMMs
        self.tc_gemm = True if tc_gemm is None else bool(tc_gemm)
        self.deliver = deliver
        self.head_idx = int(head_idx)
        self._copy_stream = None

    def _sync_weights(self):
        """Decoder weights and encoder engine from the explainer, which rebuilds them after the model's parameters were
        replaced or updated in place.  Then the decoder workspaces (prepared copies of the old weights) and the captured
        graphs (pointing at the old tensors) are dropped as well."""
        W = self.ex._grad_weights() if self.is_gradient else self.ex._lrp_weights()
        eng = self.ex.engine()
        if W is not self.W or eng is not self.eng:
            self.W, self.eng = W, eng
            self._dec_ws = {}
            self._graphs = {}

    def _requests(self, B, T, device, words_per_image=None):
        """(image, word) requests in image-major order; ``words_per_image[b]`` <= T limits image b to its own caption
        length (ragged batches: shorter captions are padded in ``tokens``, their padding words are not explained)."""
        if words_per_image is None:
            req_img = torch.arange(B, dtype=torch.int32, device=device).repeat_interleave(T)
            req_t = torch.arange(T, dtype=torch.int32, device=device).repeat(B)
            return req_img, req_t
        n = [int(v) for v in words_per_image]
        if len(n) != B or any(v < 0 or v > T for v in n):
            raise ValueError("words_per_image must hold B values in [0, T]")
        req_img = torch.tensor([b for b in range(B) for _ in range(n[b])], dtype=torch.int32, device=device)
        req_t = torch.tensor([t for b in range(B) for t in range(n[b])], dtype=torch.int32, device=device)
        return req_img, req_t

    def _run(self, imgs, tokens, req_img, req_t, heat, host=None):
        """-> (r_words, the Guided Grad-CAM operands the launches read: they must outlive a graph capturing them)"""
        est = self.eng.forward(imgs)
        r_words, _, cam = self._explain_encoded(est, self.eng.features(est, "pixel"), tokens, req_img, req_t, heat, host)
        return r_words, cam

    def _explain_encoded(self, est, feat, tokens, req_img, req_t, heat, host=None):
        """Everything after the encoder forward: explainer forward on ``feat`` (the pixel-major features of the encoder
        state ``est``), decoder kernels, relevance chain (or Grad-CAM maps) into ``heat``.  -> (r_words, the explainer
        forward's logits, Guided Grad-CAM's (maps, T, Kh, Kw) or None)."""
        st = self.ex.explainer_forward(feat, tokens)
        req_word = tokens[req_img.long(), req_t.long() + 1].to(torch.int32)       # the word each request explains
        # on the explainer's cached decoder weights: the self.W of the last _sync_weights
        r_feat, r_words = self.ex._decode(st, req_img, req_t, req_word, self.tc_gemm, self.head_idx, self._dec_ws)
        cam = None
        if self.cam == "cam":                                  # explain_cnn's (Q, P) maps: no encoder chain
            ops.grad_cam(st["feat"], r_feat, req_img, out=heat)
        elif self.cam == "guided":
            # the map expanded along y here; along x, and the product, in the first layer's epilogue of the guided chain
            fh, fw = est.feat_hw
            maps = ops.grad_cam(st["feat"], r_feat, req_img).view(-1, fh, fw)
            Kh, Kw = self.ex._expand_ops(fh, fw, int(est.x.shape[2]), int(est.x.shape[3]))
            cam = (maps, ops.cam_expand_rows(maps, Kh), Kh, Kw)
        chain = self.cam != "cam"
        fused = {} if cam is None else dict(cam=(cam[1], cam[3]))     # (TcResNetEngine has no CAM factor)
        if host is None:
            if chain:
                self.eng.relevance(est, r_feat, req_img, chunk=self.chunk, out=heat, deliver=self.deliver, **fused)
            return r_words, st["pred"], cam
        # results go to pinned host buffers: the copy of chunk i runs on a side stream under the kernels of chunk i+1
        host_heat, host_words = host
        main = torch.cuda.current_stream()
        if self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream()
        side = self._copy_stream

        def on_chunk(q0, q1):
            ev = torch.cuda.Event()
            ev.record(main)
            side.wait_event(ev)
            with torch.cuda.stream(side):
                host_heat[q0:q1].copy_(heat[q0:q1], non_blocking=True)

        side.wait_stream(main)
        with torch.cuda.stream(side):
            host_words.copy_(r_words, non_blocking=True)
            if not chain:
                host_heat.copy_(heat, non_blocking=True)
        if chain:
            self.eng.relevance(est, r_feat, req_img, chunk=self.chunk, out=heat, on_chunk=on_chunk, deliver=self.deliver,
                               **fused)
        main.wait_stream(side)
        return r_words, st["pred"], cam

    def explain(self, imgs, tokens, out=None, host_out=None, words_per_image=None):
        """imgs (B,3,H,W) fp32 (CUDA, or pinned host memory), tokens (B,T+1) long with column 0 = <start>.
        Returns (heat (Q,3,H,W) fp32, r_words (Q,T) fp32); with ``words_per_image=None`` Q = B*T and request
        q = b*T + t explains word t+1 of image b; with ragged captions (``words_per_image[b]`` words for image b,
        ``tokens`` padded to T+1) the requests are the valid (b, t) pairs in the same image-major order.
        ``host_out=(heat_host, words_host)`` (pinned tensors) additionally delivers the results to the host, the
        heat-map copy overlapped chunk by chunk with the relevance kernels.
        With ``use_graph`` the returned tensors are the graph's static outputs (overwritten by the next call)."""
        self._sync_weights()
        B, T = tokens.shape[0], tokens.shape[1] - 1
        dev = self.ex.device
        wpi = None if words_per_image is None else tuple(int(v) for v in words_per_image)
        Q = B * T if wpi is None else sum(wpi)
        shp, dt = self._heat_shape(imgs, Q)
        if Q == 0:                                               # nothing to explain
            return (torch.empty((0,) + shp[1:], device=dev, dtype=dt), torch.empty(0, T, device=dev))
        if not self.use_graph:
            imgs, tokens = imgs.to(dev, non_blocking=True), tokens.to(dev, non_blocking=True)
            req_img, req_t = self._requests(B, T, dev, wpi)
            heat = out if out is not None else torch.empty(shp, device=dev, dtype=dt)
            return heat, self._run(imgs, tokens, req_img, req_t, heat, host_out)[0]
        key = (tuple(imgs.shape), tuple(tokens.shape), wpi,
               None if host_out is None else (host_out[0].data_ptr(), host_out[1].data_ptr()))
        g = self._graphs.get(key)
        if g is None:
            s_imgs, s_toks = imgs.to(dev).clone(), tokens.to(dev).clone()
            req_img, req_t = self._requests(B, T, dev, wpi)
            heat = torch.empty(shp, device=dev, dtype=dt)
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):                       # warm-up outside capture (lazy inits, attributes)
                self._run(s_imgs, s_toks, req_img, req_t, heat, host_out)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graph = torch.cuda.CUDAGraph()
            with _graph.capture(graph):
                r_words, cam = self._run(s_imgs, s_toks, req_img, req_t, heat, host_out)
            # everything the captured kernels point at must outlive the graph (incl. the request index tensors and the
            # Guided Grad-CAM maps and operators)
            g = self._graphs[key] = (graph, s_imgs, s_toks, heat, r_words, req_img, req_t, cam)
        graph, s_imgs, s_toks, heat, r_words = g[:5]
        if imgs.is_cuda:
            s_imgs.copy_(imgs, non_blocking=True)
        else:
            self._stage_host_images(imgs, s_imgs)
        s_toks.copy_(tokens, non_blocking=True)
        graph.replay()
        return heat, r_words

    def explain_images(self, imgs, beam_size=None, max_cap_length=None, out=None, host_out=None):
        """Captions B images with the explainer's device beam search and explains every word of every caption: what
        ``explain_caption`` does for one image, for a batch.  The encoder runs once: the search reads the features of
        that pass and the explanation reuses its state, so the captions are the ones the per-image API explains (a
        search through ``model.beam_search_device`` encodes the images a second time, with the library forward).

        imgs (B,3,H,W) fp32 (CUDA, or pinned host memory).  ``beam_size`` / ``max_cap_length`` default to the
        explainer's ``CAPTION_SEARCH``, the search of its ``get_hidden_parameters``.  The requests are the (image, word)
        pairs of the captions in image-major order, as ``explain(..., words_per_image=...)`` orders them; an image whose
        caption is empty (<end> first) has none.  ``out`` (heat-maps) and ``host_out=(heat_host, words_host)`` (pinned;
        filled as ``explain`` fills them) need room for the result, which goes to their first Q rows and to the first T
        columns of ``words_host``: B * max_cap_length rows and max_cap_length columns always suffice.
        Runs eagerly even with ``use_graph``: the search replays its own CUDA graphs, and a graph of the explanation
        would be captured anew for every pattern of caption lengths.  -> ImageExplanation."""
        self._sync_weights()
        ex, dev = self.ex, self.ex.device
        beam_size = ex.CAPTION_SEARCH[0] if beam_size is None else beam_size
        max_cap_length = ex.CAPTION_SEARCH[1] if max_cap_length is None else max_cap_length
        imgs = imgs.to(dev, non_blocking=True)
        B = imgs.shape[0]
        est = self.eng.forward(imgs)
        feat = self.eng.features(est, "pixel")
        with torch.no_grad():
            proj, glob = ex._search_inputs(feat)
        captions = ex._searcher().search(proj, glob, ex.word_map, beam_size=beam_size, max_cap_length=max_cap_length)
        wpi = tuple(len(c) for c in captions)
        T, Q = max(wpi), sum(wpi)
        start = ex.word_map['<start>']
        tokens = torch.tensor([[start] + c + [0] * (T - len(c)) for c in captions], dtype=torch.long, device=dev)
        req_img, req_t = self._requests(B, T, dev, wpi)
        shp, dt = self._heat_shape(imgs, Q, est)
        if Q == 0:                                               # nothing to explain: explain's empty results
            heat, r_words = torch.empty(shp, device=dev, dtype=dt), torch.empty(0, T, device=dev)
            pred = torch.empty(B, T, ex.model.fc.out_features, device=dev)
        else:
            bufs = ([] if out is None else [out]) + ([] if host_out is None else list(host_out))
            if any(b.shape[0] < Q for b in bufs) or (host_out is not None and host_out[1].shape[1] < T):
                raise ValueError(f"out / host_out hold fewer than the {Q} requests of {T} words found")
            heat = torch.empty(shp, device=dev, dtype=dt) if out is None else out[:Q]
            host = None if host_out is None else (host_out[0][:Q], host_out[1][:Q, :T])
            r_words, pred, _ = self._explain_encoded(est, feat, tokens, req_img, req_t, heat, host)
        return ImageExplanation(captions, tokens, wpi, req_img, req_t, heat, r_words, pred)

    def _heat_shape(self, imgs, Q, est=None):
        """(shape, dtype) of Q heat-maps in the delivery format (the engine's image size is known after its first
        forward; before that it is the size of these images).  Grad-CAM: (Q, P) with P the encoder output's pixels,
        taken from the encoder state ``est`` of these images or, without one, from a forward of one image of this size
        (once per size)."""
        H, W = int(imgs.shape[2]), int(imgs.shape[3])
        if self.cam == "cam":
            if est is not None:
                self._cam_px[(H, W)] = est.feat_hw[0] * est.feat_hw[1]
            elif (H, W) not in self._cam_px:
                fh, fw = self.eng.forward(torch.zeros(1, 3, H, W, device=self.ex.device)).feat_hw
                self._cam_px[(H, W)] = fh * fw
            return (Q, self._cam_px[(H, W)]), torch.float32
        shp = (Q, H, W) if self.deliver == "channel_mean" else (Q, 3, H, W)
        return shp, (torch.float16 if self.deliver == "fp16" else torch.float32)

    def _stage_host_images(self, imgs, s_imgs):
        """Host images reach the graph's static input through one of two device staging buffers: the host->device copy
        runs on a side stream as soon as the call is made — i.e. under the kernels of the PREVIOUS step, which are still
        executing when the host has run ahead — and the main stream only pays a device-to-device copy.  A staging buffer
        is reused two calls later, after the event behind its last device-to-device copy."""
        key = tuple(s_imgs.shape)
        st = getattr(self, "_stage", None)
        if st is None or st["key"] != key:
            st = self._stage = dict(key=key, bufs=[torch.empty_like(s_imgs) for _ in range(2)],
                                    done=[None, None], n=0, stream=torch.cuda.Stream())
        k = st["n"] & 1
        st["n"] += 1
        main, side = torch.cuda.current_stream(), st["stream"]
        if st["done"][k] is not None:
            side.wait_event(st["done"][k])                  # the buffer's previous contents have been consumed
        with torch.cuda.stream(side):
            st["bufs"][k].copy_(imgs, non_blocking=True)
            arrived = torch.cuda.Event()
            arrived.record(side)
        main.wait_event(arrived)
        s_imgs.copy_(st["bufs"][k], non_blocking=True)
        st["done"][k] = torch.cuda.Event()
        st["done"][k].record(main)
