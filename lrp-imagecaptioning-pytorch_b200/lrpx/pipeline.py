"""Batched explanation pipeline: all (image, word) requests of a batch of images in one pass.

This is the throughput-oriented entry point above the reference-shaped explainers: what
``ExplainGridTDAttention.explain_caption`` does for one image (gridTDmodel.py:1141-1156: forward, then per
word decoder relevance + encoder relevance) is done here for B images x T words at once:

  encoder forward + gains (tcgen05)  ->  explainer teacher-forced forward  ->  decoder relevance kernels for
  all B*T requests  ->  encoder relevance chain (tcgen05)  ->  heat-maps (B*T,3,H,W) + r_words (B*T,T)

Optionally the whole pass is captured once into a CUDA graph (fixed B and caption length) and replayed, which
removes the launch latency of the ~2.7k small kernels of the decoder phases.
"""
import torch

from . import _graph, ops


class BatchExplainer:
    def __init__(self, explainer, chunk=128, use_graph=False, tc_gemm=None, head_idx=0, deliver="full"):
        """explainer: models.gridTDmodel.ExplainGridTDAttention, models.aoamodel.ExplainAOAAttention or
        models.adaptiveattention.ExplainAdaptiveAttention on a VGG encoder with precision 'fp32' (fp32-accurate chain)
        or 'bf16'; ``head_idx``: the attention head an AoA explanation follows (aoamodel.py:1165,
        ``explain_caption(img, head_idx)``); ``deliver``: format of the heat-maps (TcVggEngine.heat_shape): 'full' =
        fp32 (Q,3,H,W) like the reference, 'channel_mean' = fp32 (Q,H,W), 'fp16'; ``tc_gemm``: decoder GEMMs as bf16x3
        on tensor cores (default: with precision 'bf16') or on fp32 CUDA cores."""
        if not getattr(explainer, "uses_tc", False):
            raise ValueError("BatchExplainer drives the tensor-core chain: it needs a VGG-style encoder and "
                             "precision='fp32' (fp32-accurate mode) or 'bf16'")
        self.ex = explainer
        # gradient-family explainers (models/_gradient.py): same pipeline, the decoder-gradient kernels and the chain's
        # 'gradient' / 'guided' rule instead of the relevance ones
        self.is_gradient = hasattr(explainer, "_grad_weights")
        if self.is_gradient and getattr(explainer, "CAM", None):
            raise ValueError("BatchExplainer covers the gradient and guided-backpropagation explainers, not the CAM variants")
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
        self.is_aoa = hasattr(explainer, "num_head") and hasattr(explainer.model, "decoder_multihead_attention")
        self.is_adaptive = not self.is_aoa and not hasattr(explainer.model, "LanguageLSTM")   # single-LSTM decoder
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
        est = self.eng.forward(imgs)
        feat = self.eng.features(est, "pixel")
        st = self.ex.explainer_forward(feat, tokens)
        req_word = tokens[req_img.long(), req_t.long() + 1].to(torch.int32)       # the word each request explains
        if self.is_gradient and self.is_aoa:
            r_feat, r_words = ops.aoa_decoder_grad(st, self.W, self.ex.num_head, req_img, req_t, req_word,
                                                   torch.full_like(req_t, self.head_idx), tc_gemm=self.tc_gemm)
        elif self.is_gradient and self.is_adaptive:
            r_feat, r_words = ops.adaptive_decoder_grad(st, self.W, req_img, req_t, req_word, tc_gemm=self.tc_gemm)
        elif self.is_gradient:
            r_feat, r_words = ops.gridtd_decoder_grad(st, self.W, req_img, req_t, req_word,
                                                      guided=self.ex.GUIDED_DECODER, tc_gemm=self.tc_gemm)
        elif self.is_aoa:
            r_feat, r_words = ops.aoa_decoder_lrp(st, self.W, self.ex.num_head, req_img, req_t, req_word,
                                                  torch.full_like(req_t, self.head_idx), tc_gemm=self.tc_gemm,
                                                  ws_cache=self._dec_ws)
        elif self.is_adaptive:
            r_feat, r_words = ops.adaptive_decoder_lrp(st, self.W, req_img, req_t, req_word, tc_gemm=self.tc_gemm,
                                                       ws_cache=self._dec_ws)
        else:
            r_feat, r_words = ops.gridtd_decoder_lrp(st, self.W, req_img, req_t, req_word, tc_gemm=self.tc_gemm,
                                                     ws_cache=self._dec_ws)
        if host is None:
            self.eng.relevance(est, r_feat, req_img, chunk=self.chunk, out=heat, deliver=self.deliver)
            return r_words
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
        self.eng.relevance(est, r_feat, req_img, chunk=self.chunk, out=heat, on_chunk=on_chunk, deliver=self.deliver)
        main.wait_stream(side)
        return r_words

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
        # heat-map buffer in the delivery format (the engine's image size is known after its first forward; before
        # that it is the size of these images)
        H, W = int(imgs.shape[2]), int(imgs.shape[3])
        shp = (Q, H, W) if self.deliver == "channel_mean" else (Q, 3, H, W)
        dt = torch.float16 if self.deliver == "fp16" else torch.float32
        if Q == 0:                                               # nothing to explain
            return (torch.empty((0,) + shp[1:], device=dev, dtype=dt), torch.empty(0, T, device=dev))
        if not self.use_graph:
            imgs, tokens = imgs.to(dev, non_blocking=True), tokens.to(dev, non_blocking=True)
            req_img, req_t = self._requests(B, T, dev, wpi)
            heat = out if out is not None else torch.empty(shp, device=dev, dtype=dt)
            return heat, self._run(imgs, tokens, req_img, req_t, heat, host_out)
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
                r_words = self._run(s_imgs, s_toks, req_img, req_t, heat, host_out)
            # everything the captured kernels point at must outlive the graph (incl. the request index tensors)
            g = self._graphs[key] = (graph, s_imgs, s_toks, heat, r_words, req_img, req_t)
        graph, s_imgs, s_toks, heat, r_words = g[:5]
        if imgs.is_cuda:
            s_imgs.copy_(imgs, non_blocking=True)
        else:
            self._stage_host_images(imgs, s_imgs)
        s_toks.copy_(tokens, non_blocking=True)
        graph.replay()
        return heat, r_words

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
