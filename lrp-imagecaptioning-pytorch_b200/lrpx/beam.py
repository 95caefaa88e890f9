"""Beam search of the gridTD and AoA decoders on the device (SURVEY.md §8 f1).

``GridTDModel.beam_search`` (reference models/gridTDmodel.py:400-478) runs ~25 tensor ops per step and reads the
top-k result back to python lists every step.  Here a step is a fixed sequence of kernels with no host round trip:

  embedding gather + input-side GEMM -> ``lrpx_lstm_step_f32`` (AdaLSTM + sentinel gate) -> attention projections
  (library GEMM) -> ``lrpx_adaptive_attention_f32`` -> ``lrpx_lstm_step_f32`` (language LSTM) -> vocabulary GEMM ->
  ``lrpx_beam_step`` (log-softmax, top-k over the alive beams, <end> handling, compaction) ->
  ``lrpx_beam_gather_f32`` (recurrent state of the surviving beams)

over B images x k beam slots, captured into CUDA graphs of ten steps each; between two graphs the host reads the alive
counts once to stop early, and the result is read back once at the end.  Word indices equal the reference's (tests:
the reference's own beam-search fixtures, bit for bit).  ``AoaBeamSearch`` is the same loop for ``AOAModel`` /
``AOAModelBU`` (aoamodel.py:405-485): LSTM step kernel, multi-head attention and the AoA gate as library tensor ops.
"""
import math

import torch

from . import _graph, ops


class _DeviceBeamSearch:
    """The shared part: state tensors of the bookkeeping kernels, CUDA graphs of SEGMENT steps, the final pick."""
    SEGMENT = 10          # steps per CUDA graph / between two looks at the alive counts

    def __init__(self, model, use_graph=True):
        self.model = model
        self.use_graph = use_graph
        self._w = ops.WeightCache()
        self._plans = {}

    # subclasses: _weight_sources() -> tensors whose change invalidates the cache; _build_weights() -> dict;
    # _alloc(R, P, f) -> dict of step tensors; _step(t, w) -> logits tensor name is t["logits"]; _pairs(t) -> gather
    # pairs; _prepare(t, B, k, feats, glob, w)
    def _weights(self):
        # the captured graphs hold raw pointers: every tensor a step reads belongs to the key, so that a model moved or
        # re-loaded after the first search gets fresh plans
        m = self.model

        def build():
            self._plans = {}
            return self._build_weights()
        return self._w.get(self._weight_sources(), build,
                           tuple(t.data_ptr() for t in (m.embedding.weight, m.fc.weight, m.fc.bias)))   # read in place: pointer only

    def _plan(self, B, k, L, P, start_id, end_id):
        key = (B, k, L, P, start_id, end_id)
        pl = self._plans.get(key)
        if pl is not None:
            return pl
        m, w = self.model, self._weights()
        dev = m.fc.weight.device
        R = B * k
        f = lambda *s: torch.zeros(*s, device=dev, dtype=torch.float32)
        i32 = lambda *s: torch.zeros(*s, device=dev, dtype=torch.int32)
        t = self._alloc(R, P, f)
        t.update(logits=f(R, m.vocab_size), scores=f(B, k), comp_scores=f(B, k), n_alive=i32(B), n_comp=i32(B),
                 seqs=i32(B, k, L + 1), comp_seqs=i32(B, k, L + 1), comp_len=i32(B, k), src_row=i32(R),
                 prev=torch.zeros(R, device=dev, dtype=torch.int64))
        recurrent = self._recurrent(t)
        pairs = self._pairs(t)

        def run(s0, s1):
            if s0 == 0:
                for x in recurrent + [t[n] for n in ("scores", "comp_scores", "n_comp", "comp_len", "seqs", "comp_seqs")]:
                    x.zero_()
                t["n_alive"].fill_(k)
                t["prev"].fill_(start_id)
                t["seqs"][:, :, 0] = start_id
            for step in range(s0, s1):
                self._step(t, w)
                ops.beam_step(t["logits"], t["scores"], t["n_alive"], t["seqs"], t["comp_seqs"], t["comp_len"],
                              t["comp_scores"], t["n_comp"], t["prev"], t["src_row"], step, end_id)
                ops.beam_gather(t["src_row"], pairs)

        # the loop runs in segments of SEGMENT steps; between two segments the host looks at n_alive once and stops when
        # every beam of every image has ended (the reference's `if unfinished_num == 0: break`, gridTDmodel.py:453-454)
        segs = [(s0, min(L, s0 + self.SEGMENT)) for s0 in range(0, L, self.SEGMENT)]
        graphs = None
        if self.use_graph:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side), torch.no_grad():     # warm-up outside capture (lazy library initialisation)
                run(0, min(L, 2))
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graphs = []
            for s0, s1 in segs:
                g = torch.cuda.CUDAGraph()
                with _graph.capture(g), torch.no_grad():
                    run(s0, s1)
                graphs.append(g)
        pl = self._plans[key] = (t, run, segs, graphs)
        return pl

    def _search(self, B, P, feats, glob, word_map, beam_size, max_cap_length):
        w = self._weights()
        k, L = int(beam_size), int(max_cap_length)
        t, run, segs, graphs = self._plan(B, k, L, P, word_map['<start>'], word_map['<end>'])
        with torch.no_grad():
            self._prepare(t, B, k, feats, glob, w)
            for n, (s0, s1) in enumerate(segs):
                if n and not bool(t["n_alive"].any()):           # one small read-back per segment
                    break
                if graphs is not None:
                    graphs[n].replay()
                else:
                    run(s0, s1)
            n_comp, comp_len, comp_scores = t["n_comp"].tolist(), t["comp_len"].tolist(), t["comp_scores"].tolist()
            comp_seqs, seqs = t["comp_seqs"].tolist(), t["seqs"][:, 0].tolist()
        special = {word_map['<start>'], word_map['<end>'], word_map['<unk>'], word_map['<pad>']}
        out = []
        for b in range(B):
            if n_comp[b] > 0:                                   # best completed sequence, first one on ties (:463-465)
                sc = comp_scores[b][:n_comp[b]]
                j = sc.index(max(sc))
                seq = comp_seqs[b][j][:comp_len[b][j]]
            else:
                seq = seqs[b][:min(L + 1, 20)]                  # seqs[0][:20] (:467)
            out.append([wd for wd in seq if wd not in special])
        return out


class GridTDBeamSearch(_DeviceBeamSearch):
    """model: models.gridTDmodel.GridTDModel or GridTDModelBU on a CUDA device (eval mode: dropout is identity)."""

    def _weight_sources(self):
        m = self.model
        cell, L, xg, hg, att = m.AdaLSTM.lstm_cell, m.LanguageLSTM, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate, m.AdaAttention
        return [cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh, xg.weight, xg.bias, hg.weight, hg.bias,
                L.weight_ih, L.weight_hh, L.bias_ih, L.bias_hh, att.W_g_proj.weight, att.W_s_proj.weight,
                att.W_s_proj.bias, att.w_h.weight]

    def _build_weights(self):
        m = self.model
        cell, L, xg, hg, att = m.AdaLSTM.lstm_cell, m.LanguageLSTM, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate, m.AdaAttention
        H, E, K = m.hidden_dim, m.embed_dim, att.num_pixel
        dev = cell.weight_ih.device
        # x1 = [h2 | glob | emb] (:431): recurrent rows [h2 | h1] -> (4H gates | sentinel gate)
        W1_rec = torch.cat((torch.cat((cell.weight_ih[:, :H], cell.weight_hh), 1),
                            torch.cat((xg.weight[:, :H], hg.weight), 1)), 0).t().contiguous()      # (2H, 5H)
        W1_in = torch.cat((cell.weight_ih[:, H:], xg.weight[:, H:]), 0).t().contiguous()           # (2E, 5H)
        b1 = torch.cat((cell.bias_ih + cell.bias_hh, xg.bias + hg.bias)).contiguous()
        W2 = torch.cat((L.weight_ih, L.weight_hh), 1).t().contiguous()                             # (3H, 4H)
        Wa = torch.zeros(2 * H, 2 * K, device=dev)
        Wa[:H, :K] = att.W_g_proj.weight.t()
        Wa[H:, K:] = att.W_s_proj.weight.t()
        return dict(W1p=ops.lstm_prep_weights(W1_rec, 5), W1_glob=W1_in[:E].contiguous(), W1_emb=W1_in[E:].contiguous(),
                    b1=b1, W2p=ops.lstm_prep_weights(W2, 4), b2=(L.bias_ih + L.bias_hh).contiguous(), Wa=Wa,
                    ba=torch.cat((torch.zeros(K, device=dev), att.W_s_proj.bias)),
                    w_h=att.w_h.weight.reshape(-1).contiguous(), fcW_t=m.fc.weight.t())

    def _alloc(self, R, P, f):
        m = self.model
        H, E, K = m.hidden_dim, m.embed_dim, m.AdaAttention.num_pixel
        return dict(A=f(R, P, H), img_proj=f(R, P, K), preg=f(R, 5 * H),                      # per-call inputs
                    hcat=f(R, 2 * H), x2c=f(R, 3 * H), hs=f(R, 2 * H), c1=f(R, H), c2=f(R, H),
                    h1n=f(R, H), c1n=f(R, H), h2n=f(R, H), c2n=f(R, H), g=f(R, H), i=f(R, H), f=f(R, H), st=f(R, H),
                    ctx=f(R, H), ctx_hat=f(R, H), alpha=f(R, P), beta=f(R), emb=f(R, E), pre1=f(R, 5 * H),
                    hsp=f(R, 2 * K), xo=f(R, H))

    def _recurrent(self, t):
        return [t["hcat"], t["x2c"], t["c1"], t["c2"]]

    def _pairs(self, t):
        H = self.model.hidden_dim
        return [(t["hcat"][:, :H], t["h2n"]), (t["hcat"][:, H:], t["h1n"]), (t["x2c"][:, 2 * H:], t["h2n"]),
                (t["c1"], t["c1n"]), (t["c2"], t["c2n"])]

    def _step(self, t, w):
        m = self.model
        H = m.hidden_dim
        torch.index_select(m.embedding.weight, 0, t["prev"], out=t["emb"])
        torch.addmm(t["preg"], t["emb"], w["W1_emb"], out=t["pre1"])
        ops.lstm_step(t["hcat"], w["W1p"], t["pre1"], 5, t["c1"], t["h1n"], t["c1n"], t["g"], t["i"], t["f"],
                      s=t["st"], h_copy1=t["x2c"][:, H:2 * H], h_copy2=t["hs"][:, :H], s_copy=t["hs"][:, H:])
        torch.addmm(w["ba"], t["hs"], w["Wa"], out=t["hsp"])
        ops.adaptive_attention(t["A"], t["img_proj"], t["hsp"], w["w_h"], t["st"], t["ctx"], t["ctx_hat"],
                               t["alpha"], t["beta"], ctx_hat_copy=t["x2c"][:, :H])
        ops.lstm_step(t["x2c"], w["W2p"], w["b2"], 4, t["c2"], t["h2n"], t["c2n"], t["g"], t["i"], t["f"])
        torch.add(t["ctx_hat"], t["h2n"], out=t["xo"])
        torch.addmm(m.fc.bias, t["xo"], w["fcW_t"], out=t["logits"])

    def _prepare(self, t, B, k, A, glob, w):
        m = self.model
        P, H = A.shape[1], A.shape[2]
        t["A"].view(B, k, P, H).copy_(A.unsqueeze(1).expand(B, k, P, H))
        t["img_proj"].view(B, k, P, -1).copy_(m.AdaAttention.W_v_proj(A).unsqueeze(1).expand(B, k, P, -1))
        preg = torch.addmm(w["b1"], glob.float(), w["W1_glob"])                       # (B,5H)
        t["preg"].view(B, k, -1).copy_(preg.unsqueeze(1).expand(B, k, -1))

    def search(self, image_feature_proj, global_img_feature, word_map, beam_size=3, max_cap_length=20):
        """image_feature_proj (B, hidden, P) and global_img_feature (B, embed) as ``GridTDModel._encode`` returns them.
        -> list of B token lists ``sen_idx`` (special tokens removed, reference :466-468)."""
        if not image_feature_proj.is_cuda:
            raise ops._lib.LrpxError("GridTDBeamSearch needs CUDA tensors: lrpx has no CPU fallback")
        B, H, P = image_feature_proj.shape
        return self._search(B, P, image_feature_proj.transpose(1, 2), global_img_feature, word_map, beam_size,
                            max_cap_length)


class AoaBeamSearch(_DeviceBeamSearch):
    """model: models.aoamodel.AOAModel or AOAModelBU on a CUDA device.  A step (aoamodel.py:118-122, :54-108):
    LSTM over [emb | glob] (``lrpx_lstm_step_f32``, input-side half as one GEMM), q projection, scaled dot-product
    attention of 8 heads over the image's keys / values, sigmoid(gate(h)) * linear(ctx), vocabulary GEMM."""

    def _weight_sources(self):
        m = self.model
        L, mha = m.LanguageLSTM, m.decoder_multihead_attention
        return [L.weight_ih, L.weight_hh, L.bias_ih, L.bias_hh, mha.q_proj.weight, mha.q_proj.bias,
                m.decoder_aoa_linear_gate.weight, m.decoder_aoa_linear_gate.bias, m.decoder_aoa_linear.weight,
                m.decoder_aoa_linear.bias]

    def _build_weights(self):
        m = self.model
        L, mha = m.LanguageLSTM, m.decoder_multihead_attention
        E = m.embed_dim
        return dict(Wp=ops.lstm_prep_weights(L.weight_hh.t().contiguous(), 4), W_emb=L.weight_ih[:, :E].t().contiguous(),
                    W_glob=L.weight_ih[:, E:].t().contiguous(), b=(L.bias_ih + L.bias_hh).contiguous(),
                    Wq_t=mha.q_proj.weight.t(), Wg_t=m.decoder_aoa_linear_gate.weight.t(),
                    Wl_t=m.decoder_aoa_linear.weight.t(), fcW_t=m.fc.weight.t())

    def _alloc(self, R, P, f):
        m = self.model
        H, E, nh = m.hidden_dim, m.embed_dim, m.num_head
        dk = H // nh
        return dict(keyT=f(R, nh, dk, P), val=f(R, nh, P, dk), preg=f(R, 4 * H),                # per-call inputs
                    hin=f(R, H), c=f(R, H), hn=f(R, H), cn=f(R, H), g=f(R, H), i=f(R, H), f=f(R, H), emb=f(R, E),
                    pre=f(R, 4 * H), q=f(R, H), sc=f(R, nh, 1, P), ctx=f(R, nh, 1, dk), gate=f(R, H), lin=f(R, H),
                    xo=f(R, H))

    def _recurrent(self, t):
        return [t["hin"], t["c"]]

    def _pairs(self, t):
        return [(t["hin"], t["hn"]), (t["c"], t["cn"])]

    def _step(self, t, w):
        m = self.model
        H, nh = m.hidden_dim, m.num_head
        dk = H // nh
        mha = m.decoder_multihead_attention
        R = t["hin"].shape[0]
        torch.index_select(m.embedding.weight, 0, t["prev"], out=t["emb"])
        torch.addmm(t["preg"], t["emb"], w["W_emb"], out=t["pre"])
        ops.lstm_step(t["hin"], w["Wp"], t["pre"], 4, t["c"], t["hn"], t["cn"], t["g"], t["i"], t["f"])
        torch.addmm(mha.q_proj.bias, t["hn"], w["Wq_t"], out=t["q"])
        torch.matmul(t["q"].view(R, nh, 1, dk), t["keyT"], out=t["sc"])
        t["sc"].div_(math.sqrt(dk))
        alpha = torch.softmax(t["sc"], dim=-1)
        torch.matmul(alpha, t["val"], out=t["ctx"])
        torch.addmm(m.decoder_aoa_linear_gate.bias, t["hn"], w["Wg_t"], out=t["gate"])
        torch.addmm(m.decoder_aoa_linear.bias, t["ctx"].view(R, H), w["Wl_t"], out=t["lin"])
        torch.addcmul(t["hn"], torch.sigmoid(t["gate"]), t["lin"], out=t["xo"])          # context_aoa + ht (:122)
        torch.addmm(m.fc.bias, t["xo"], w["fcW_t"], out=t["logits"])

    def _prepare(self, t, B, k, proj, glob, w):
        m = self.model
        P, H = proj.shape[1], proj.shape[2]
        nh = m.num_head
        dk = H // nh
        key = m.decoder_k_proj(proj).view(B, P, nh, dk).permute(0, 2, 3, 1)              # (B, heads, dk, P)
        val = m.decoder_v_proj(proj).view(B, P, nh, dk).transpose(1, 2)                  # (B, heads, P, dk)
        t["keyT"].view(B, k, nh, dk, P).copy_(key.unsqueeze(1).expand(B, k, nh, dk, P))
        t["val"].view(B, k, nh, P, dk).copy_(val.unsqueeze(1).expand(B, k, nh, P, dk))
        preg = torch.addmm(w["b"], glob.float(), w["W_glob"])                            # (B,4H)
        t["preg"].view(B, k, -1).copy_(preg.unsqueeze(1).expand(B, k, -1))

    def search(self, image_feature_proj, global_img_feature, word_map, beam_size=3, max_cap_length=20):
        """image_feature_proj (B, P, hidden) and global_img_feature (B, hidden) as ``AOAModel._encode`` returns them."""
        if not image_feature_proj.is_cuda:
            raise ops._lib.LrpxError("AoaBeamSearch needs CUDA tensors: lrpx has no CPU fallback")
        B, P, H = image_feature_proj.shape
        return self._search(B, P, image_feature_proj, global_img_feature, word_map, beam_size, max_cap_length)


class AdaptiveBeamSearch(_DeviceBeamSearch):
    """model: models.adaptiveattention.AdaptiveAttentionCaptioningModel on a CUDA device.  A step
    (adaptiveattention.py:128-135): AdaLSTM over [emb | glob] with the sentinel gate from the old hidden state
    (``lrpx_lstm_step_f32``, five gates), adaptive attention (``lrpx_adaptive_attention_f32``), fc(ctx_hat + h)."""

    def _weight_sources(self):
        m = self.model
        cell, xg, hg, att = m.AdaLSTM.lstm_cell, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate, m.AdaAttention
        return [cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh, xg.weight, xg.bias, hg.weight, hg.bias,
                att.W_g_proj.weight, att.W_s_proj.weight, att.W_s_proj.bias, att.w_h.weight]

    def _build_weights(self):
        m = self.model
        cell, xg, hg, att = m.AdaLSTM.lstm_cell, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate, m.AdaAttention
        H, E, K = m.hidden_dim, m.embed_dim, att.num_pixel
        dev = cell.weight_ih.device
        W_rec = torch.cat((cell.weight_hh, hg.weight), 0).t().contiguous()             # (H, 5H)
        W_in = torch.cat((cell.weight_ih, xg.weight), 0).t().contiguous()              # (2E, 5H): rows [emb ; glob]
        Wa = torch.zeros(2 * H, 2 * K, device=dev)
        Wa[:H, :K] = att.W_g_proj.weight.t()
        Wa[H:, K:] = att.W_s_proj.weight.t()
        return dict(Wp=ops.lstm_prep_weights(W_rec, 5), W_emb=W_in[:E].contiguous(), W1_glob=W_in[E:].contiguous(),
                    b1=torch.cat((cell.bias_ih + cell.bias_hh, xg.bias + hg.bias)).contiguous(), Wa=Wa,
                    ba=torch.cat((torch.zeros(K, device=dev), att.W_s_proj.bias)),
                    w_h=att.w_h.weight.reshape(-1).contiguous(), fcW_t=m.fc.weight.t())

    def _alloc(self, R, P, f):
        m = self.model
        H, E, K = m.hidden_dim, m.embed_dim, m.AdaAttention.num_pixel
        return dict(A=f(R, P, H), img_proj=f(R, P, K), preg=f(R, 5 * H),                   # per-call inputs
                    hin=f(R, H), c=f(R, H), hs=f(R, 2 * H), hn=f(R, H), cn=f(R, H), g=f(R, H), i=f(R, H), f=f(R, H), st=f(R, H),
                    ctx=f(R, H), ctx_hat=f(R, H), alpha=f(R, P), beta=f(R), emb=f(R, E), pre=f(R, 5 * H),
                    hsp=f(R, 2 * K), xo=f(R, H))

    def _recurrent(self, t):
        return [t["hin"], t["c"]]

    def _pairs(self, t):
        return [(t["hin"], t["hn"]), (t["c"], t["cn"])]

    def _step(self, t, w):
        m = self.model
        H = m.hidden_dim
        torch.index_select(m.embedding.weight, 0, t["prev"], out=t["emb"])
        torch.addmm(t["preg"], t["emb"], w["W_emb"], out=t["pre"])
        ops.lstm_step(t["hin"], w["Wp"], t["pre"], 5, t["c"], t["hn"], t["cn"], t["g"], t["i"], t["f"],
                      s=t["st"], h_copy2=t["hs"][:, :H], s_copy=t["hs"][:, H:])
        torch.addmm(w["ba"], t["hs"], w["Wa"], out=t["hsp"])
        ops.adaptive_attention(t["A"], t["img_proj"], t["hsp"], w["w_h"], t["st"], t["ctx"], t["ctx_hat"],
                               t["alpha"], t["beta"])
        torch.add(t["ctx_hat"], t["hn"], out=t["xo"])
        torch.addmm(m.fc.bias, t["xo"], w["fcW_t"], out=t["logits"])

    _prepare = GridTDBeamSearch._prepare

    def search(self, image_feature_proj, global_img_feature, word_map, beam_size=3, max_cap_length=20):
        """image_feature_proj (B, hidden, P) and global_img_feature (B, embed) as the model's ``_encode`` returns them."""
        if not image_feature_proj.is_cuda:
            raise ops._lib.LrpxError("AdaptiveBeamSearch needs CUDA tensors: lrpx has no CPU fallback")
        B, H, P = image_feature_proj.shape
        return self._search(B, P, image_feature_proj.transpose(1, 2), global_img_feature, word_map, beam_size,
                            max_cap_length)
