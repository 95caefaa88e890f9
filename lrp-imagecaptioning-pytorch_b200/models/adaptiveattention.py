"""Host-side mirror of the LRP entry points of the reference's models/adaptiveattention.py (SURVEY.md §8 f2).

* ``AdaptiveAttentionCaptioningModel`` — state_dict-compatible module (reference :101-121) with ``forward``
  (:137-190), ``beam_search`` (:370-447) and ``greedy_search`` (:449-489).
* ``ExplainAdaptiveAttention`` — ``get_hidden_parameters`` (:626-677), ``forward_greedy`` (:567-624),
  ``explain_caption_wordt`` (:679-771), ``explain_cnn`` (:773-777), ``explain_caption`` (:779-794),
  ``lrp_linear_eps`` (:525-546).

The decoder relevance of all requested words is ONE call of ``lrpx_adaptive_decoder_lrp_f32``; the explainer's
teacher-forced forward runs on the fused step kernels (``lrpx_lstm_step_f32`` with the sentinel gate as fifth gate,
``lrpx_adaptive_attention_f32``); the encoder relevance is the tcgen05 chain (VGG, bf16) or the fp32 rule kernels.
"""
import torch
import torch.nn as nn

from LRPtools import utils as LRPutil
from lrpx import ops
from lrpx import decoder as _dec
from models.gridTDmodel import AdaptiveAttention, AdaptiveLSTMCell, Encoder, ExplainGridTDAttention

__all__ = ["Encoder", "AdaptiveLSTMCell", "AdaptiveAttention", "AdaptiveAttentionCaptioningModel",
           "ExplainAdaptiveAttention"]


class AdaptiveAttentionCaptioningModel(nn.Module):
    """reference :101-489 (the surface the explainer and evaluation.py use)."""
    EPS = LRPutil.EPSILON

    def __init__(self, embed_dim, hidden_dim, vocab_size, encoder_type, n_pixel=196):
        super().__init__()
        self.embed_dim = embed_dim
        self.hidden_dim = hidden_dim
        self.vocab_size = vocab_size
        self.encoder_type = encoder_type
        self.dropout = nn.Dropout(0.5)
        self.img_encoder = Encoder(self.encoder_type)
        self.encoder_raw_dim = self.img_encoder.feat_dim
        self.img_projector = nn.Conv2d(self.encoder_raw_dim, self.hidden_dim, kernel_size=1, stride=1)
        self.global_img_feature_proj = nn.Linear(self.encoder_raw_dim, self.embed_dim)
        self.AdaLSTM = AdaptiveLSTMCell(embed_dim * 2, hidden_dim)
        self.AdaAttention = AdaptiveAttention(self.hidden_dim, n_pixel)
        self.embedding = nn.Embedding(vocab_size, embed_dim)
        self.fc = nn.Linear(hidden_dim, vocab_size)
        self.relu = nn.ReLU()

    def init_hidden_state(self, V):
        h = torch.zeros(V.shape[0], self.hidden_dim, device=V.device)
        return h, torch.zeros_like(h)

    def predict_next_word(self, image_feature_proj, xt, states):
        """reference :128-135"""
        ht, ct = states
        ht, ct, st = self.AdaLSTM(xt, (ht, ct))
        context_t_hat, context_t, alpha_t, beta_t = self.AdaAttention(image_feature_proj, ht, st)
        predict_score_t = self.fc(self.dropout(context_t_hat + ht))
        return predict_score_t, alpha_t, beta_t, (ht, ct)

    def _encode(self, images):
        batch_size = images.size(0)
        image_features, avg_feature = self.img_encoder(images)
        image_feature_proj = self.relu(self.img_projector(image_features)).contiguous().view(batch_size, self.hidden_dim, -1)
        global_img_feature = self.relu(self.global_img_feature_proj(avg_feature))
        if global_img_feature.dim() == 1:
            global_img_feature = global_img_feature.unsqueeze(0)
        return image_features, image_feature_proj, global_img_feature

    def forward(self, images, encoded_captions, caption_lengths, ss_prob=None):
        """Teacher-forced forward (reference :137-190; scheduled sampling is not part of the LRP path)."""
        if ss_prob is not None:
            raise NotImplementedError("scheduled sampling is outside the LRP hot path (SURVEY.md §2 #9)")
        batch_size = images.size(0)
        _, image_feature_proj, global_img_feature = self._encode(images)
        num_pixels = image_feature_proj.size(-1)
        state = self.init_hidden_state(image_feature_proj)
        max_length = int(max(caption_lengths)) - 1
        predictions = torch.zeros(batch_size, max_length, self.vocab_size, device=images.device)
        alphas = torch.zeros(batch_size, max_length, num_pixels, device=images.device)
        betas = torch.zeros(batch_size, max_length, 1, device=images.device)
        last_scores = None
        for t in range(max_length):
            xt = torch.cat((self.embedding(encoded_captions[:, t]), global_img_feature), dim=-1)
            predict_score_t, alpha_t, beta_t, state = self.predict_next_word(image_feature_proj, xt, state)
            predictions[:, t, :] = predict_score_t
            alphas[:, t, :] = alpha_t
            betas[:, t, :] = beta_t
            last_scores = torch.log_softmax(predict_score_t, -1)
        return predictions, alphas, betas, last_scores, max_length

    def beam_search(self, imgs, word_map, beam_size=3, max_cap_length=20):
        """reference :370-447 (batch size 1).  ``beam_idx`` uses floor division — the reference's true division
        (:414) is an IndexError on torch >= 1.6 (Q8).  No bad-ending removal in this model (:444-446)."""
        self.eval()
        assert imgs.size(0) == 1
        rev_word_map = {v: k for k, v in word_map.items()}
        vocab_size = len(word_map)
        dev = imgs.device
        complete_seqs, complete_seqs_scores = [], []
        with torch.no_grad():
            k_prev_words = torch.full((beam_size, 1), word_map['<start>'], dtype=torch.long, device=dev)
            top_k_scores = torch.zeros(beam_size, 1, device=dev)
            seqs = k_prev_words.clone()
            _, image_feature_proj, global_img_feature = self._encode(imgs)
            image_feature_proj = image_feature_proj.expand(beam_size, *image_feature_proj.size()[1:])
            global_img_feature = global_img_feature.expand(beam_size, global_img_feature.size(-1))
            state = self.init_hidden_state(image_feature_proj)
            unfinished_num = beam_size
            for step in range(max_cap_length):
                xt = torch.cat((self.embedding(k_prev_words).squeeze(1), global_img_feature), dim=-1)
                predict_score_t, _, _, state = self.predict_next_word(image_feature_proj, xt, state)
                scores = top_k_scores.expand((unfinished_num, vocab_size)) + torch.log_softmax(predict_score_t, dim=-1)
                if step == 0:
                    top_k_scores, top_words = scores[0].topk(beam_size, -1, True, True)
                else:
                    top_k_scores, top_words = scores.view(-1).topk(unfinished_num, -1, True, True)
                beam_idx = top_words // vocab_size
                next_word_idx = top_words % vocab_size
                seqs = torch.cat([seqs[beam_idx], next_word_idx.unsqueeze(1)], dim=1)
                nw = next_word_idx.tolist()
                incomplete_inds = [i for i, w in enumerate(nw) if w != word_map['<end>']]
                complete_inds = [i for i, w in enumerate(nw) if w == word_map['<end>']]
                if complete_inds:
                    complete_seqs.extend(seqs[complete_inds].tolist())
                    complete_seqs_scores.extend(top_k_scores[complete_inds].tolist())
                unfinished_num -= len(complete_inds)
                if unfinished_num == 0:
                    break
                seqs = seqs[incomplete_inds]
                keep = beam_idx[incomplete_inds]
                state = tuple(s[keep] for s in state)
                image_feature_proj = image_feature_proj[keep]
                global_img_feature = global_img_feature[keep]
                top_k_scores = top_k_scores[incomplete_inds].unsqueeze(1)
                k_prev_words = next_word_idx[incomplete_inds].unsqueeze(1)
            if complete_seqs:
                seq = complete_seqs[complete_seqs_scores.index(max(complete_seqs_scores))]
            else:
                seq = seqs[0][:20].tolist()
            special = {word_map['<start>'], word_map['<end>'], word_map['<unk>'], word_map['<pad>']}
            sen_idx = [w for w in seq if w not in special]
            return [' '.join(rev_word_map[w] for w in sen_idx)], sen_idx

    def beam_search_device(self, imgs, word_map, beam_size=3, max_cap_length=20):
        """``beam_search`` with the step loop on the device (lrpx.beam.AdaptiveBeamSearch) for B >= 1 images at once;
        same word indices.  -> (sentence, sen_idx) for one image, a list of such pairs for a batch."""
        from lrpx.beam import AdaptiveBeamSearch
        self.eval()
        if getattr(self, "_beam", None) is None:
            self._beam = AdaptiveBeamSearch(self)
        with torch.no_grad():
            _, image_feature_proj, global_img_feature = self._encode(imgs)
        rev_word_map = {v: k for k, v in word_map.items()}
        out = [([' '.join(rev_word_map[w] for w in idx)], idx)
               for idx in self._beam.search(image_feature_proj, global_img_feature, word_map, beam_size, max_cap_length)]
        return out[0] if len(out) == 1 else out

    def greedy_search(self, imgs, word_map, max_cap_length=20):
        """reference :449-489 -> (sentences, token lists incl. <start>; finished rows continue with <pad>=0)."""
        self.eval()
        batch_size = imgs.size(0)
        rev_word_map = {v: k for k, v in word_map.items()}
        with torch.no_grad():
            k_prev_words = torch.zeros(batch_size, max_cap_length, dtype=torch.long, device=imgs.device)
            k_prev_words[:, 0] = word_map['<start>']
            _, image_feature_proj, global_img_feature = self._encode(imgs)
            state = self.init_hidden_state(image_feature_proj)
            unfinished = None
            for step in range(max_cap_length - 1):
                xt = torch.cat((self.embedding(k_prev_words[:, step]), global_img_feature), dim=-1)
                predict_score_t, _, _, state = self.predict_next_word(image_feature_proj, xt, state)
                top_words = torch.log_softmax(predict_score_t, dim=-1).topk(1, -1, True, True)[1]
                not_end = top_words != word_map['<end>']
                unfinished = not_end if unfinished is None else unfinished & not_end
                k_prev_words[:, step + 1] = (top_words * unfinished.type_as(top_words))[:, 0]
            seqs = k_prev_words.tolist()
        special = {word_map['<start>'], word_map['<end>'], word_map['<unk>'], word_map['<pad>']}
        sentences = [' '.join(rev_word_map[w] for w in s if w not in special) for s in seqs]
        return sentences, seqs


class ExplainAdaptiveAttention(ExplainGridTDAttention):
    """reference :491-848.  Shares the encoder handling, request batching and result bookkeeping of
    ExplainGridTDAttention; the saved state and the decoder rule are this model's own."""

    def __init__(self, args, word_map, model=None, precision=None):
        self._common_init(args, word_map, model, precision,
                          lambda: AdaptiveAttentionCaptioningModel(args.embed_dim, args.hidden_dim, len(word_map),
                                                                   args.encoder))
        m = self.model
        if m.embed_dim != m.hidden_dim:
            # the reference's saved x_t is embed_dim + hidden_dim wide but holds [emb | glob] = 2 * embed_dim (:636,:663)
            raise ValueError("ExplainAdaptiveAttention needs embed_dim == hidden_dim (reference :636)")
        self.adalstm_weight_i, self.adalstm_weight_h = m.AdaLSTM.lstm_cell.weight_ih, m.AdaLSTM.lstm_cell.weight_hh
        self.adalstm_bias_i, self.adalstm_bias_h = m.AdaLSTM.lstm_cell.bias_ih, m.AdaLSTM.lstm_cell.bias_hh

    _LRP_WEIGHTS = staticmethod(_dec.adaptive_weights)

    def _explainer_weights(self):
        """[W_hh ; h_gate] (recurrent, in the step kernel's layout), [W_ih ; x_gate] (input side), summed biases;
        cached until a parameter changes."""
        m = self.model
        cell, xg, hg = m.AdaLSTM.lstm_cell, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate

        def build():
            W_rec = torch.cat((cell.weight_hh, hg.weight), 0).t().contiguous()          # (H, 5H)
            W_in = torch.cat((cell.weight_ih, xg.weight), 0).t().contiguous()           # (2E, 5H)
            b = torch.cat((cell.bias_ih + cell.bias_hh, xg.bias + hg.bias)).contiguous()
            return ops.lstm_prep_weights(W_rec, 5), W_in, b
        return self._caches["expl_w"].get([cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh, xg.weight, xg.bias,
                                           hg.weight, hg.bias], build)

    def explainer_forward(self, feat, tokens, quirk_double_bias_ih=None, want_gates=False):
        """(``quirk_double_bias_ih`` is accepted for the shared gradient-family plumbing and has no effect: this model's
        explainers add both LSTM biases, reference :554-565, :883.  ``want_gates`` also saves the output gate and the
        sentinel gate, the state of the gradient explainers, reference :941-960.)
        The explainer's teacher-forced forward (reference :631-677) batched over images.  feat: (B,P,C) pixel-major
        encoder output; tokens: (B,L) long, column 0 = <start>.  Returns the saved state in the layout of
        lrpx_adaptive_args, T = L-1 steps.  Per step: ``lrpx_lstm_step_f32`` (4 gates + sentinel gate from h_t, the
        input-side halves precomputed for all steps), one library GEMM for both attention projections,
        ``lrpx_adaptive_attention_f32``."""
        if not feat.is_cuda:
            raise ops._lib.LrpxError("explainer_forward needs CUDA tensors: lrpx has no CPU fallback")
        m = self.model
        B, P, C = feat.shape
        H, E = m.hidden_dim, m.embed_dim
        T = tokens.shape[1] - 1
        dev = feat.device
        att = m.AdaAttention
        K = att.num_pixel
        new = lambda *shape: torch.empty(*shape, device=dev, dtype=torch.float32)
        with torch.no_grad():
            feat = feat.contiguous()
            avg = feat.mean(1)
            # every GEMM of this forward runs on the tcgen05 kernels (ops.LinearX3: bf16x3, fp32 accuracy)
            ipw = m.img_projector.weight
            z_proj = self._lx("proj", ipw, None, lambda: (ipw.detach().reshape(H, C), None))(feat.view(B * P, C)).view(B, P, H)   # without bias (:762)
            A = (z_proj + m.img_projector.bias).clamp(min=0).contiguous()
            z_glob = self._lx("glob", m.global_img_feature_proj.weight)(avg)       # without bias (:745)
            glob = (z_glob + m.global_img_feature_proj.bias).clamp(min=0)
            img_proj = self._lx("wv", att.W_v_proj.weight, att.W_v_proj.bias)(A.view(B * P, H)).view(B, P, K)   # (B,P,K)
            Wrec_p, W_in, b = self._explainer_weights()
            att_lin = self._attention_layer()
            w_h = att.w_h.weight.reshape(-1).contiguous()
            emb = m.embedding(tokens[:, :T])                                                     # (B,T,E)
            x = torch.cat((emb, glob.unsqueeze(1).expand(B, T, E)), -1).contiguous()             # (B,T,2E)  :649
            cell, xg, hg = m.AdaLSTM.lstm_cell, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate
            pre = self._lx("pre", [cell.weight_ih, xg.weight], [cell.bias_ih, cell.bias_hh, xg.bias, hg.bias],
                           lambda: (W_in.t().contiguous(), b))(x.transpose(0, 1).reshape(T * B, 2 * E)).view(T, B, 5 * H)
            h, c = torch.zeros(B, T + 1, H, device=dev), torch.zeros(B, T + 1, H, device=dev)
            g, i, f, st, ctx, ctx_hat = (new(B, T, H) for _ in range(6))
            alpha, beta = new(B, T, P), new(B, T)
            og, sg = (new(B, T, H), new(B, T, H)) if want_gates else (None, None)
            # the step kernel reads every column of its input rows in every CTA while its CTAs write the new state:
            # the recurrent input is ping-ponged between two copies
            hin = torch.zeros(2, B, H, device=dev)
            hs = new(B, 2 * H)                                # [h_{t+1} | s_t]
            for t in range(T):
                p, q = t & 1, (t & 1) ^ 1
                ops.lstm_step(hin[p], Wrec_p, pre[t], 5, c[:, t], h[:, t + 1], c[:, t + 1], g[:, t], i[:, t], f[:, t],
                              s=st[:, t], h_copy0=hin[q], h_copy2=hs[:, :H], s_copy=hs[:, H:],
                              o=None if og is None else og[:, t], sg=None if sg is None else sg[:, t])
                hsp = att_lin(hs)                                                                 # (B,2K)
                ops.adaptive_attention(A, img_proj, hsp, w_h, st[:, t], ctx[:, t], ctx_hat[:, t], alpha[:, t],
                                       beta[:, t])
            pred = self._lx("fc", m.fc.weight, m.fc.bias)((ctx_hat + h[:, 1:]).view(B * T, H)).view(B, T, -1)
        out = dict(x=x, h=h, c=c, g=g, i=i, f=f, st=st, ctx=ctx, ctx_hat=ctx_hat, alpha=alpha, beta=beta, pred=pred,
                   feat=feat, avg=avg, z_proj=z_proj.contiguous(), A=A, z_glob=z_glob)
        if want_gates:
            out.update(o=og, sg=sg)
        return out

    # ------------------------------------------------------------------ reference entry points
    CAPTION_SEARCH = (3, 20)              # get_hidden_parameters, reference :626-677

    _BEAM = "AdaptiveBeamSearch"
    _REMOVE_BAD_ENDINGS = False           # this model's beam search keeps the sentence as it is (:444-446)

    def _expose_state(self, st):
        """attributes the reference exposes (:634-646)"""
        self.predictions, self.alphas, self.betas = st["pred"][0], st["alpha"][0], st["beta"][0]
        self.xt, self.ht, self.ct = st["x"][0], st["h"][0], st["c"][0]
        self.gt, self.it_act, self.ft_act = st["g"][0], st["i"][0], st["f"][0]
        self.st, self.context, self.context_hat = st["st"][0], st["ctx"][0], st["ctx_hat"][0]
        self.avg_feature = st["avg"][0]

    def _decode(self, st, req_img, req_t, req_word, tc_gemm, head_idx=0, ws_cache=None):
        return ops.adaptive_decoder_lrp(st, self._lrp_weights(), req_img, req_t, req_word, tc_gemm=tc_gemm,
                                        ws_cache=ws_cache)


# ================================================================================================ gradient family (f4)
from models._gradient import GradientFamily      # noqa: E402


def adaptive_grad_weights(sd):
    """B operands of lrpx_adaptive_grad_args from an AdaptiveAttentionCaptioningModel state_dict."""
    H = sd["fc.weight"].shape[1]
    return {
        "W_g": torch.cat((sd["AdaLSTM.lstm_cell.weight_ih"], sd["AdaLSTM.lstm_cell.weight_hh"]), 1).contiguous(),   # (4H, 2E+H)
        "W_fc": sd["fc.weight"].contiguous(),
        "W_glob": sd["global_img_feature_proj.weight"].contiguous(),
        "W_proj": sd["img_projector.weight"].reshape(H, -1).contiguous(),
    }


class ExplainAdaptiveGradient(GradientFamily, ExplainAdaptiveAttention):
    """reference :851-1095: gradient of the word's logit through the single-LSTM adaptive-attention decoder (attention and
    sentinel split applied at the explained step only, :987-994) and the image encoder."""
    EX_TYPE = 'gradient'

    def __init__(self, args, word_map, model=None, precision=None):
        ExplainAdaptiveAttention.__init__(self, args, word_map, model=model, precision=precision)
        self._check_encoder()

    _GRAD_WEIGHTS = staticmethod(adaptive_grad_weights)

    def _expose_state(self, st):
        ExplainAdaptiveAttention._expose_state(self, st)
        self.ot_act, self.sen_gate = st["o"][0], st["sg"][0]

    def _decode(self, st, req_img, req_t, req_word, tc_gemm, head_idx=0, ws_cache=None):
        return ops.adaptive_decoder_grad(st, self._grad_weights(), req_img, req_t, req_word, tc_gemm=tc_gemm)


class ExplainiAdaptiveGuidedGradient(ExplainAdaptiveGradient):
    """reference :1098-1216 (the class name's typo is the reference's): the decoder half equals the plain gradient's (its
    masks compare ReLU outputs with `< 0`), the encoder half is guided backpropagation."""
    EX_TYPE = 'GuidedBackpropagate'
    RULE = "guided"


class ExplainAdaptiveGradCam(ExplainAdaptiveGradient):
    """reference :1218-1259."""
    EX_TYPE = 'GradCam'
    CAM = "cam"


class ExplainAdaptiveGuidedGradCam(ExplainiAdaptiveGuidedGradient):
    """reference :1261-1325."""
    EX_TYPE = 'GuidedGradCam'
    CAM = "guided"
