"""Host-side mirror of the LRP entry points of the reference's models/aoamodel.py.

* ``AOAModel`` — state_dict-compatible module (reference :111-139): ``forward`` (:160-211), ``beam_search``
  (:405-485), tuner entry points ``get_lrp_weight_step`` (:597-626), ``forwardlrp_context`` (:628-677),
  ``sample_lrp`` (:679-745).
* ``ExplainAOAAttention`` — ``get_hidden_parameters`` (:990-1062), ``lrp_mha`` (:812-862),
  ``explain_caption_wordt(t, head_idx)`` (:1064-1156), ``explain_cnn`` (:1158-1163), ``explain_caption``
  (:1165-1181), ``explain_caption_words`` (:1183-1194).

The relevance arithmetic runs in liblrpx.so (``lrpx_aoa_decoder_lrp_f32``, ``lrpx_fc_lrp_weights_f32``, the
encoder kernels); see models/gridTDmodel.py for the shared conventions.
"""
import math

import torch
import torch.nn as nn

from LRPtools import lrp_wrapper
from LRPtools import utils as LRPutil
from lrpx import ops
from lrpx import decoder as _dec
from models.gridTDmodel import (BAD_ENDINGS, STOP_WORDS, Encoder, ExplainGridTDAttention, GridTDModel,  # noqa: F401
                                _lstm_forward)


class Add(nn.Module):
    def forward(self, x, y):
        return x + y


class MultiHeadedDotAttention(nn.Module):
    """reference :54-108.  The decoder instantiates it with project_k_v_flag=False, norm_q=False, aoa=False."""

    def __init__(self, num_head, hidden_dim, dropout=0.3, project_k_v_flag=True, norm_q=True, aoa=True):
        super().__init__()
        assert hidden_dim % num_head == 0
        self.d_k = hidden_dim // num_head
        self.num_head = num_head
        self.norm = nn.BatchNorm1d(hidden_dim, track_running_stats=True) if norm_q else (lambda x: x)
        self.q_proj = nn.Linear(hidden_dim, hidden_dim)
        if project_k_v_flag:
            self.k_proj = nn.Linear(hidden_dim, hidden_dim)
            self.v_proj = nn.Linear(hidden_dim, hidden_dim)
        else:
            self.k_proj = lambda x: x
            self.v_proj = lambda x: x
        self.aoa = aoa
        if aoa:
            self.aoa_layer = nn.Sequential(nn.Linear(2 * hidden_dim, 2 * hidden_dim), nn.GLU())
            self.add = Add()
        self.dropout = nn.Dropout(p=dropout)

    def forward(self, query, key, value):
        single_query = query.dim() == 2
        if single_query:
            query = query.unsqueeze(1)
        bs = query.size(0)
        query = self.norm(query.transpose(1, 2)).transpose(1, 2)
        q = self.q_proj(query).view(bs, -1, self.num_head, self.d_k).transpose(1, 2)
        k = self.k_proj(key).view(bs, -1, self.num_head, self.d_k).transpose(1, 2)
        v = self.v_proj(value).view(bs, -1, self.num_head, self.d_k).transpose(1, 2)
        scores = torch.matmul(q, k.transpose(-2, -1)) / math.sqrt(self.d_k)
        alpha = torch.softmax(scores, dim=-1)
        p = nn.functional.dropout(alpha, 0.1) if self.training else alpha
        x = torch.matmul(p, v).transpose(1, 2).contiguous().view(bs, -1, self.num_head * self.d_k)
        if self.aoa:
            x = self.add(self.aoa_layer(self.dropout(torch.cat([x, query], -1))), query)
        if single_query:
            x, alpha = x.squeeze(1), alpha.squeeze(2)       # alpha: (bs, heads, P)
        return x, alpha


class AOAModel(nn.Module):
    """reference :111-745 (the LRP-related surface)."""
    EPS = LRPutil.EPSILON

    def __init__(self, embed_dim, hidden_dim, num_head, vocab_size, encoder_type):
        super().__init__()
        self.embed_dim, self.hidden_dim, self.vocab_size = embed_dim, hidden_dim, vocab_size
        self.encoder_type, self.num_head = encoder_type, num_head
        if hidden_dim % num_head != 0:
            raise TypeError("the number of head should be dividable by the hidden dim")
        self.dropout = nn.Dropout(0.3)
        self.img_encoder = Encoder(self.encoder_type)
        self.encoder_raw_dim = self.img_encoder.feat_dim
        self.img_projector = nn.Conv2d(self.encoder_raw_dim, self.hidden_dim, kernel_size=1, stride=1)
        self.embedding = nn.Embedding(vocab_size, embed_dim)
        self.LanguageLSTM = nn.LSTMCell(hidden_dim + embed_dim, hidden_dim)
        self.decoder_k_proj = nn.Linear(hidden_dim, hidden_dim)
        self.decoder_v_proj = nn.Linear(hidden_dim, hidden_dim)
        self.decoder_multihead_attention = MultiHeadedDotAttention(num_head=num_head, hidden_dim=hidden_dim,
                                                                   project_k_v_flag=False, norm_q=False, aoa=False)
        self.decoder_aoa_linear_gate = nn.Linear(hidden_dim, hidden_dim)
        self.decoder_aoa_linear = nn.Linear(hidden_dim, hidden_dim)
        self.fc = nn.Linear(hidden_dim, vocab_size)
        self.relu = nn.ReLU()
        self._stop_cache = {}

    init_hidden_state = GridTDModel.init_hidden_state
    remove_bad_endings = GridTDModel.remove_bad_endings
    sample_next_word = GridTDModel.sample_next_word
    lrp_linear_eps = GridTDModel.lrp_linear_eps
    _stop_mask = GridTDModel._stop_mask

    def _encode(self, images):
        bs = images.size(0)
        image_features, _ = self.img_encoder(images)
        before = self.img_projector(image_features)
        proj = self.relu(before).contiguous().view(bs, self.hidden_dim, -1).transpose(1, 2)     # (bs, P, H)
        return image_features, proj, torch.mean(proj, dim=1)

    def _attend(self, ht, key, value):
        context, alpha_t = self.decoder_multihead_attention(ht, key, value)
        gate = self.decoder_aoa_linear_gate(ht)
        lin = self.decoder_aoa_linear(context)
        return torch.sigmoid(gate) * lin, alpha_t

    def predict_next_word(self, image_feature_proj, xt, states):
        ht, ct = self.LanguageLSTM(xt, states)
        context_aoa, alpha_t = self._attend(ht, self.decoder_k_proj(image_feature_proj),
                                            self.decoder_v_proj(image_feature_proj))
        return self.fc(self.dropout(context_aoa + ht)), alpha_t, None, (ht, ct)

    def greedy_search(self, imgs, word_map, max_cap_length=20):
        """reference :487-530 -> (sentences with the bad endings removed, token lists incl. <start>).  (The reference
        returns the filtered word list of the LAST image as its second value; the token lists of all rows are returned
        here, like its gridTD sibling.)"""
        self.eval()
        rev_word_map = {v: k for k, v in word_map.items()}
        with torch.no_grad():
            k_prev_words = torch.zeros(imgs.size(0), max_cap_length, dtype=torch.long, device=imgs.device)
            k_prev_words[:, 0] = word_map['<start>']
            _, proj, glob = self._encode(imgs)
            state = self.init_hidden_state(proj)
            unfinished = None
            for step in range(max_cap_length - 1):
                xt = torch.cat((self.embedding(k_prev_words[:, step]), glob), dim=-1)
                predict_score_t, _, _, state = self.predict_next_word(proj, xt, state)
                top_words = torch.log_softmax(predict_score_t, dim=-1).topk(1, -1, True, True)[1]
                not_end = top_words != word_map['<end>']
                unfinished = not_end if unfinished is None else unfinished & not_end
                k_prev_words[:, step + 1] = (top_words * unfinished.type_as(top_words))[:, 0]
            seqs = k_prev_words.tolist()
        special = {word_map['<start>'], word_map['<end>'], word_map['<unk>'], word_map['<pad>']}
        sentences = [' '.join(rev_word_map[w] for w in s if w not in special) for s in seqs]
        return self.remove_bad_endings(sentences), seqs

    def forward(self, images, encoded_captions, caption_lengths, ss_prob=None):
        if ss_prob is not None:
            raise NotImplementedError("scheduled sampling is outside the LRP hot path (SURVEY.md §2 #9)")
        _, proj, glob = self._encode(images)
        state = self.init_hidden_state(proj)
        max_length = int(max(caption_lengths)) - 1
        preds, last_scores = [], None
        for t in range(max_length):
            xt = torch.cat((self.embedding(encoded_captions[:, t]), glob), dim=-1)
            score, _, _, state = self.predict_next_word(proj, xt, state)
            preds.append(score)
            last_scores = torch.log_softmax(score, -1)
        return torch.stack(preds, 1), None, None, last_scores, max_length

    def beam_search(self, imgs, word_map, beam_size=3, max_cap_length=20):
        """reference :405-485 (batch size 1)."""
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
            _, proj, glob = self._encode(imgs)
            proj = proj.expand(beam_size, *proj.size()[1:])
            glob = glob.expand(beam_size, glob.size(-1))
            state = self.init_hidden_state(proj)
            unfinished_num = beam_size
            for step in range(max_cap_length):
                xt = torch.cat((self.embedding(k_prev_words).squeeze(1), glob), dim=-1)
                score, _, _, state = self.predict_next_word(proj, xt, state)
                scores = top_k_scores.expand((unfinished_num, vocab_size)) + torch.log_softmax(score, dim=-1)
                if step == 0:
                    top_k_scores, top_words = scores[0].topk(beam_size, -1, True, True)
                else:
                    top_k_scores, top_words = scores.view(-1).topk(unfinished_num, -1, True, True)
                beam_idx = top_words // vocab_size
                next_word_idx = top_words % vocab_size
                seqs = torch.cat([seqs[beam_idx], next_word_idx.unsqueeze(1)], dim=1)
                nw = next_word_idx.tolist()
                incomplete = [i for i, w in enumerate(nw) if w != word_map['<end>']]
                complete = [i for i, w in enumerate(nw) if w == word_map['<end>']]
                if complete:
                    complete_seqs.extend(seqs[complete].tolist())
                    complete_seqs_scores.extend(top_k_scores[complete].tolist())
                unfinished_num -= len(complete)
                if unfinished_num == 0:
                    break
                seqs = seqs[incomplete]
                keep = beam_idx[incomplete]
                state = tuple(s[keep] for s in state)
                proj, glob = proj[keep], glob[keep]
                top_k_scores = top_k_scores[incomplete].unsqueeze(1)
                k_prev_words = next_word_idx[incomplete].unsqueeze(1)
            if complete_seqs:
                seq = complete_seqs[complete_seqs_scores.index(max(complete_seqs_scores))]
            else:
                seq = seqs[0][:20].tolist()
            special = {word_map['<start>'], word_map['<end>'], word_map['<unk>'], word_map['<pad>']}
            sen_idx = [w for w in seq if w not in special]
            return self.remove_bad_endings([' '.join(rev_word_map[w] for w in sen_idx)]), sen_idx

    def sample(self, images, word_map, caption_lengths, opt={}):
        """reference aoamodel.py:206-245 -> (seq, seq_logprobs, max_length), see GridTDModel.sample."""
        batch_size = images.size(0)
        sample_method = opt.get('sample_method', 'greedy')
        temperature = opt.get('temperature', 1.0)
        max_length = int(max(caption_lengths)) - 1
        _, proj, glob = self._encode(images)
        state = self.init_hidden_state(proj)
        dev = proj.device
        seq = torch.zeros(batch_size, max_length, dtype=torch.long, device=dev)
        seq_logprobs = torch.zeros(batch_size, max_length, device=dev)
        it = torch.full((batch_size,), word_map['<start>'], dtype=torch.long, device=dev)
        unfinished = None
        for t in range(max_length):
            xt = torch.cat((self.embedding(it), glob), dim=-1)
            score, _, _, state = self.predict_next_word(proj, xt, state)
            it, sample_logprobs = self.sample_next_word(torch.log_softmax(score, dim=-1), sample_method, temperature)
            finished = it == word_map['<end>']
            unfinished = ~finished if unfinished is None else unfinished & ~finished
            it = it * unfinished.type_as(it)
            seq[:, t] = it
            seq_logprobs[:, t] = sample_logprobs.view(-1)
            if int(unfinished.sum()) == 0:
                break
        return seq, seq_logprobs, max_length

    def beam_search_device(self, imgs, word_map, beam_size=3, max_cap_length=20):
        """``beam_search`` with the step loop on the device (lrpx.beam.AoaBeamSearch) for B >= 1 images at once; same
        word indices.  -> (sentence, sen_idx) for one image, a list of such pairs for a batch."""
        from lrpx.beam import AoaBeamSearch
        self.eval()
        if getattr(self, "_beam", None) is None:
            self._beam = AoaBeamSearch(self)
        with torch.no_grad():
            _, proj, glob = self._encode(imgs)
        rev_word_map = {v: k for k, v in word_map.items()}
        out = [(self.remove_bad_endings([' '.join(rev_word_map[w] for w in idx)]), idx)
               for idx in self._beam.search(proj, glob, word_map, beam_size, max_cap_length)]
        return out[0] if len(out) == 1 else out

    # ------------------------------------------------------------------ lrp_tune
    def get_lrp_weight_step(self, predictions_t, rev_word_map, ht_, context_aoa):
        """reference :597-626 -> (weight_of_context_aoa, weight_of_ht); one batched kernel."""
        with torch.no_grad():
            w_ctx, w_h, _ = ops.fc_lrp_weights(predictions_t.detach(), ht_.detach(), context_aoa.detach(),
                                               self.fc.weight.detach(), self._stop_mask(rev_word_map, predictions_t.device))
        return w_ctx, w_h

    def _tune_step(self, glob, key, value, word_embedding, state):
        L = self.LanguageLSTM
        xt_ = torch.cat((word_embedding, glob), dim=-1)
        h_, c_, _, _, _ = _lstm_forward(xt_, state[0], state[1], L.weight_ih, L.weight_hh, L.bias_ih, L.bias_hh)
        context_aoa_, _ = self._attend(h_, key, value)
        return context_aoa_, (h_, c_)

    def forwardlrp_context(self, images, encoded_captions, caption_lengths, rev_word_map):
        """reference :628-677 (dropout on both projections, Q7)."""
        _, proj, glob = self._encode(images)
        key, value = self.decoder_k_proj(proj), self.decoder_v_proj(proj)
        state = self.init_hidden_state(proj)
        max_length = int(max(caption_lengths)) - 1
        predictions, weighted = [], []
        for t in range(max_length):
            context_aoa_, state = self._tune_step(glob, key, value, self.embedding(encoded_captions[:, t]), state)
            h_ = state[0]
            score = self.fc(self.dropout(context_aoa_ + h_))
            w_ctx, w_h = self.get_lrp_weight_step(score, rev_word_map, h_, context_aoa_)
            predictions.append(score)
            weighted.append(self.fc(self.dropout(w_ctx * context_aoa_ + h_ * w_h)))
        return torch.stack(predictions, 1), torch.stack(weighted, 1), max_length

    def sample_lrp(self, images, rev_word_map, word_map, caption_lengths, opt={}):
        """reference :679-745; the LRP step sees the log-softmax scores as forward output (:725-727, Q7)."""
        bs = images.size(0)
        sample_method = opt.get('sample_method', 'greedy')
        temperature = opt.get('temperature', 1.0)
        max_length = int(max(caption_lengths)) - 1
        _, proj, glob = self._encode(images)
        key, value = self.decoder_k_proj(proj), self.decoder_v_proj(proj)
        state = self.init_hidden_state(proj)
        dev = images.device
        seq = torch.zeros(bs, max_length, dtype=torch.long, device=dev)
        seq_logprobs = torch.zeros(bs, max_length, device=dev)
        it = torch.full((bs,), word_map['<start>'], dtype=torch.long, device=dev)
        unfinished = None
        for t in range(max_length):
            context_aoa_, state = self._tune_step(glob, key, value, self.embedding(it), state)
            h_ = state[0]
            score = torch.log_softmax(self.fc(self.dropout(context_aoa_ + h_)), dim=-1)
            w_ctx, w_h = self.get_lrp_weight_step(score, rev_word_map, h_, context_aoa_)
            logp = torch.log_softmax(self.fc(context_aoa_ * w_ctx + w_h * h_), dim=-1)
            it, sample_logprobs = self.sample_next_word(logp, sample_method, temperature)
            finished = it == word_map['<end>']
            unfinished = ~finished if unfinished is None else unfinished & ~finished
            it = it * unfinished.type_as(it)
            seq[:, t] = it
            seq_logprobs[:, t] = sample_logprobs.view(-1)
            if int(unfinished.sum()) == 0:
                break
        return seq, seq_logprobs, max_length


class AOAModelBU(AOAModel):
    """reference :1779-2400 — the AoA decoder on bottom-up region features (B, 36, 2048): ``Linear(2048, hidden)``
    projector (:1797), global feature = mean of the projected regions (:1845).  ``beam_search`` (:2059-2135, default
    length 30), ``get_lrp_weight_step`` (:2235-2264), ``forwardlrp_context`` (:2266-2310) and ``sample_lrp``
    (:2312-2400) are the parent's code over ``_encode``."""

    def __init__(self, embed_dim, hidden_dim, num_head, vocab_size, encoder_type):
        nn.Module.__init__(self)
        self.embed_dim, self.hidden_dim, self.vocab_size = embed_dim, hidden_dim, vocab_size
        self.encoder_type, self.num_head = encoder_type, num_head
        if hidden_dim % num_head != 0:
            raise TypeError("the number of head should be dividable by the hidden dim")
        self.dropout = nn.Dropout(0.3)
        self.encoder_raw_dim = 2048
        self.img_projector = nn.Linear(self.encoder_raw_dim, self.hidden_dim)
        self.embedding = nn.Embedding(vocab_size, embed_dim)
        self.LanguageLSTM = nn.LSTMCell(hidden_dim + embed_dim, hidden_dim)
        self.decoder_k_proj = nn.Linear(hidden_dim, hidden_dim)
        self.decoder_v_proj = nn.Linear(hidden_dim, hidden_dim)
        self.decoder_multihead_attention = MultiHeadedDotAttention(num_head=num_head, hidden_dim=hidden_dim,
                                                                   project_k_v_flag=False, norm_q=False, aoa=False)
        self.decoder_aoa_linear_gate = nn.Linear(hidden_dim, hidden_dim)
        self.decoder_aoa_linear = nn.Linear(hidden_dim, hidden_dim)
        self.fc = nn.Linear(hidden_dim, vocab_size)
        self.relu = nn.ReLU()
        self._stop_cache = {}

    def _encode(self, images_features):
        proj = self.relu(self.img_projector(images_features)).contiguous()     # (bs, regions, hidden)
        return images_features, proj, torch.mean(proj, dim=1)

    def beam_search(self, images_features, word_map, beam_size=3, max_cap_length=30):
        return AOAModel.beam_search(self, images_features, word_map, beam_size, max_cap_length)

    def beam_search_device(self, images_features, word_map, beam_size=3, max_cap_length=30):
        return AOAModel.beam_search_device(self, images_features, word_map, beam_size, max_cap_length)


class ExplainAOAAttention(ExplainGridTDAttention):
    """reference :748-1254."""

    def __init__(self, args, word_map, model=None, precision=None):
        self.rev_word_map = {v: k for k, v in word_map.items()}
        self.num_head = args.num_head
        self._common_init(args, word_map, model, precision,
                          lambda: AOAModel(args.embed_dim, args.hidden_dim, args.num_head, len(word_map), args.encoder))
        self.model.decoder_multihead_attention.eval()

    def _lrp_weights(self):
        key = ops.weight_stamp(self.model.parameters())           # rebuilt after an update of the model's parameters
        if self._weights is None or self._weights_key != key:
            self._weights = _dec.aoa_weights({k: v.detach() for k, v in self.model.state_dict().items()})
            self._weights_key = key
        return self._weights

    def _explainer_weights(self, quirk_double_bias_ih=True):
        """Recurrent weights in the step kernel's layout, input-side weights and summed biases; cached until a
        parameter changes."""
        L = self.model.LanguageLSTM
        src = [L.weight_ih, L.weight_hh, L.bias_ih, L.bias_hh]
        key = (quirk_double_bias_ih,) + tuple((t.data_ptr(), t._version) for t in src)
        if getattr(self, "_expl_w_key", None) != key:
            with torch.no_grad():
                lb2 = L.bias_ih if quirk_double_bias_ih else L.bias_hh                    # Q3 (:873)
                self._expl_w = (ops.lstm_prep_weights(L.weight_hh.t().contiguous(), 4), L.weight_ih.t().contiguous(),
                                (L.bias_ih + lb2).contiguous())
            self._expl_w_key = key
        return self._expl_w

    def explainer_forward(self, feat, tokens, quirk_double_bias_ih=True, want_gates=False):
        """The explainer's teacher-forced forward (reference :999-1062) batched over images; returns the saved
        state in the layout of lrpx_aoa_args.  Q3: the LSTM adds bias_ih twice (:873).  ``want_gates`` also saves the
        output gate ``o`` (the gradient explainers' state, reference :1371).

        The AoA decoder feeds nothing of the attention back into its LSTM (x_t = [emb_t | glob], :1030), so only the
        recurrence is sequential: T launches of ``lrpx_lstm_step_f32`` writing h, c, g, i, f straight into the (B,T,.)
        state tensors (the input-side half of the gates is one GEMM over all steps), then query projection, 8-head
        attention, AoA gate / linear and the vocabulary projection ONCE over all B*T positions.  CUDA only
        (tests/helpers.py holds the step-by-step tensor-op restatement this is checked against)."""
        if not feat.is_cuda:
            raise ops._lib.LrpxError("explainer_forward needs CUDA tensors: lrpx has no CPU fallback")
        m = self.model
        B, P, C = feat.shape
        H, E = m.hidden_dim, m.embed_dim
        T = tokens.shape[1] - 1
        nh, dk = m.num_head, H // m.num_head
        dev = feat.device
        with torch.no_grad():
            feat = feat.contiguous()
            # every GEMM of this forward runs on the tcgen05 kernels (ops.LinearX3: bf16x3, fp32 accuracy)
            ipw = m.img_projector.weight
            A_pre = self._lx("proj", ipw, m.img_projector.bias,
                             lambda: (ipw.detach().reshape(H, C), m.img_projector.bias.detach()))(feat.view(B * P, C)).view(B, P, H)
            A = A_pre.clamp(min=0)
            glob = A.mean(1)
            A2 = A.view(B * P, H)
            key = self._lx("k", m.decoder_k_proj.weight, m.decoder_k_proj.bias)(A2).view(B, P, H)
            value = self._lx("v", m.decoder_v_proj.weight, m.decoder_v_proj.bias)(A2).view(B, P, H)
            kT = key.view(B, P, nh, dk).permute(0, 2, 3, 1)                      # (B,nh,dk,P)
            vh = value.view(B, P, nh, dk).transpose(1, 2)                        # (B,nh,P,dk)
            mha = m.decoder_multihead_attention
            Wp_hh, W_in, b = self._explainer_weights(quirk_double_bias_ih)
            x = torch.cat((m.embedding(tokens[:, :T]), glob.unsqueeze(1).expand(B, T, H)), -1).contiguous()   # (B,T,E+H)
            pre = self._lx("pre", W_in, b, lambda: (W_in.t().contiguous(), b))(x.transpose(0, 1).reshape(T * B, E + H)).view(T, B, 4 * H)
            h, c = torch.zeros(B, T + 1, H, device=dev), torch.zeros(B, T + 1, H, device=dev)
            g, i, f = (torch.empty(B, T, H, device=dev) for _ in range(3))
            o = torch.empty(B, T, H, device=dev) if want_gates else None
            hin = torch.zeros(2, B, H, device=dev)           # the step kernel's input rows, ping-ponged over the steps
            for t in range(T):
                p, q = t & 1, (t & 1) ^ 1
                ops.lstm_step(hin[p], Wp_hh, pre[t], 4, c[:, t], h[:, t + 1], c[:, t + 1], g[:, t], i[:, t], f[:, t],
                              h_copy0=hin[q], o=None if o is None else o[:, t])
            hn = h[:, 1:]                                                         # (B,T,H)
            hn2 = hn.reshape(B * T, H)
            qv = self._lx("q", mha.q_proj.weight, mha.q_proj.bias)(hn2).view(B, T, nh, dk).transpose(1, 2)   # (B,nh,T,dk)
            alpha = torch.softmax(torch.matmul(qv, kT) / math.sqrt(dk), dim=-1)   # (B,nh,T,P)
            ctx = torch.matmul(alpha, vh).transpose(1, 2).reshape(B, T, H)
            gate = self._lx("gate", m.decoder_aoa_linear_gate.weight, m.decoder_aoa_linear_gate.bias)(hn2).view(B, T, H)
            lin = self._lx("lin", m.decoder_aoa_linear.weight, m.decoder_aoa_linear.bias)(ctx.reshape(B * T, H)).view(B, T, H)
            caoa = torch.sigmoid(gate) * lin
            pred = self._lx("fc", m.fc.weight, m.fc.bias)((caoa + hn).reshape(B * T, H)).view(B, T, m.vocab_size)
            st = dict(x=x, g=g, i=i, f=f, ctx=ctx.contiguous(), caoa=caoa.contiguous(), caoa_lin=lin.contiguous(),
                      caoa_gate=gate.contiguous(), alpha=alpha.transpose(1, 2).contiguous(), pred=pred, h=h, c=c,
                      feat=feat, A_pre=A_pre.contiguous(), A=A.contiguous(), glob=glob, key=key,
                      value=value.contiguous())
            if want_gates:
                st["o"] = o
        return st

    _BEAM = "AoaBeamSearch"

    def _search_inputs(self, feat):
        m = self.model
        B, P, C = feat.shape
        Wp = m.img_projector.weight.reshape(m.hidden_dim, -1)
        proj = torch.addmm(m.img_projector.bias, feat.reshape(B * P, C), Wp.t()).clamp(min=0).view(B, P, -1)   # (B,P,H)
        return proj, proj.mean(1)

    def get_hidden_parameters(self, img_filepath):
        self.img = self.preprocess_img(img_filepath)
        enc = self._find_caption(img_filepath, beam_size=3, max_cap_length=20)
        self._set_state(self.img, self.beam_caption_encode, enc)

    def forward_greedy(self, img_filepath):
        """reference :883-950: the saved state for the beam-size-1 caption."""
        self.img = self.preprocess_img(img_filepath)
        enc = self._find_caption(img_filepath, beam_size=1, max_cap_length=20)
        self._set_state(self.img, self.beam_caption_encode, enc)

    def _set_state(self, img, tokens, enc=None):
        if self._empty_caption(tokens):
            return
        feat, (fh, fw), est = enc if enc is not None else self.encode_images(img)
        toks = torch.tensor([tokens], dtype=torch.long, device=self.device)
        st = self.explainer_forward(feat, toks)
        self._state, self._enc_state, self._feat_hw = st, est, (fh, fw)
        self.caption_length = len(tokens) - 1
        self.num_pixels = feat.shape[1]
        self.predictions, self.alphas = st["pred"][0], st["alpha"][0]
        self.xt, self.ht, self.ct = st["x"][0], st["h"][0], st["c"][0]
        self.gt, self.it_act, self.ft_act = st["g"][0], st["i"][0], st["f"][0]
        self.context, self.context_aoa = st["ctx"][0], st["caoa"][0]
        self.context_aoa_linear, self.context_aoa_gate = st["caoa_lin"][0], st["caoa_gate"][0]
        self.key, self.value = st["key"], st["value"]
        self.image_features = feat[0].t().reshape(1, feat.shape[2], fh, fw)

    def _decoder_lrp(self, ts, head_idx):
        toks = self.beam_caption_encode
        dev = self.device
        i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=dev)
        return ops.aoa_decoder_lrp(self._state, self._lrp_weights(), self.num_head, i32([0] * len(ts)), i32(list(ts)),
                                   i32([toks[t + 1] for t in ts]), i32([head_idx] * len(ts)),
                                   tc_gemm=(self.precision in ('bf16', 'mixed')))

    def lrp_mha(self, alpha, value, r_context, context, head_idx):
        """reference :812-862 (same argument order): relevance of the values of ONE head (others get 0, Q5).
        alpha (heads,P), value (P,H), r_context / context (1,H) or (H,) -> (P,H), on the device
        (``lrpx_lrp_mha_f32``; CUDA tensors only).  explain_caption_wordt runs the fused decoder kernel."""
        return ops.lrp_mha(alpha, value, r_context, context, self.num_head, head_idx)

    def explain_caption_wordt(self, t, head_idx):
        """reference :1064-1156 -> (r_img_feature (1,C,h,w), r_words (t+1,))."""
        assert t < self.caption_length
        r_feat, r_words = self._decoder_lrp([t], head_idx)
        fh, fw = self._feat_hw
        return r_feat[0].t().reshape(1, -1, fh, fw), r_words[0, :t + 1]

    def explain_caption(self, img_filepath, head_idx, t_list=None):
        """reference :1165-1181."""
        self.img_filepath = img_filepath
        self.get_hidden_parameters(img_filepath)
        T = self.caption_length
        if T == 0:
            return [], []
        r_feat, r_words = self._decoder_lrp(list(range(T)), head_idx)
        if self.uses_tc:
            heat = self.engine().relevance(self._enc_state, r_feat, torch.zeros(T, dtype=torch.int32, device=self.device))
        else:
            enc = self.model.img_encoder.encoder
            lrp_wrapper.add_lrp(enc)
            fh, fw = self._feat_hw
            heat = torch.cat([lrp_wrapper.compute_lrp(enc, self.img.detach().clone(), precision='simt',
                                                      target=r_feat[t].t().reshape(1, -1, fh, fw)) for t in range(T)])
        if self.ACCUMULATE_LIKE_REFERENCE:
            heat = torch.cumsum(heat, 0)
        relevance_imgs = [heat[t:t + 1] for t in range(T)]
        relevance_preceeding_words = [r_words[t, :t + 1] for t in range(T)]
        self.save_linguistic_explanation(relevance_preceeding_words)
        return relevance_imgs, relevance_preceeding_words

    def explain_region_features(self, images_features, head_idx, beam_size=3, t_list=None):
        """BASELINE config 3: the AoA decoder on bottom-up region features (1, 36, 2048) with ``AOAModelBU`` —
        beam search (reference :2059-2135), the explainer's teacher-forced forward (:999-1062) and the decoder
        relevance (:1064-1156) down to the region features, where the explanation ends (there is no CNN).
        The reference has no ``Explain*BU`` class (SURVEY.md §8c(ii)); this is ``explain_caption`` without
        ``explain_cnn``.  -> (list of (1, regions, 2048) relevances, list of (t+1,) word relevances), one per word."""
        feats = images_features.to(self.device).float()
        assert feats.dim() == 3 and feats.size(0) == 1
        # the caption search runs on the device (same word indices) unless the model's beam_search was replaced
        search = (self.model.beam_search_device if self.DEVICE_BEAM_SEARCH and 'beam_search' not in self.model.__dict__
                  else self.model.beam_search)
        self.beam_caption, self.beam_caption_encode = search(feats, self.word_map, beam_size=beam_size)
        self.beam_caption_encode = [self.word_map['<start>']] + self.beam_caption_encode
        toks = torch.tensor([self.beam_caption_encode], dtype=torch.long, device=self.device)
        st = self.explainer_forward(feats, toks)
        self._state, self._enc_state, self._feat_hw = st, None, (feats.shape[1], 1)
        self.caption_length = len(self.beam_caption_encode) - 1
        self.num_pixels = feats.shape[1]
        self.predictions, self.alphas = st["pred"][0], st["alpha"][0]
        ts = list(range(self.caption_length)) if t_list is None else list(t_list)
        r_feat, r_words = self._decoder_lrp(ts, head_idx)
        return [r_feat[k:k + 1] for k in range(len(ts))], [r_words[k, :t + 1] for k, t in enumerate(ts)]

    def explain_region_features_batch(self, images_features, head_idx, beam_size=3, tokens=None):
        """BASELINE config 3 for B feature sets at once: one batched device beam search (``beam_search_device``), one
        batched explainer forward over the padded captions, ONE decoder-relevance launch sequence over all (image, word)
        requests.  ``tokens`` ((B, L) long, column 0 = <start>, 0-padded) skips the search.
        -> (r_feat (Q, regions, 2048), r_words (Q, T), req_img (Q,), req_t (Q,), captions: list of B token lists)."""
        feats = images_features.to(self.device).float().contiguous()
        B = feats.shape[0]
        if tokens is None:
            found = self.model.beam_search_device(feats, self.word_map, beam_size=beam_size)
            caps = [found[1]] if B == 1 else [c[1] for c in found]
        else:
            caps = [[int(w) for w in row[1:] if int(w) != 0] for row in tokens.tolist()]
        T = max(1, max(len(c) for c in caps))
        start = self.word_map['<start>']
        toks = torch.tensor([[start] + c + [0] * (T - len(c)) for c in caps], dtype=torch.long, device=self.device)
        st = self.explainer_forward(feats, toks)
        i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=self.device)
        req_img = i32([b for b in range(B) for _ in caps[b]])
        req_t = i32([t for b in range(B) for t in range(len(caps[b]))])
        req_word = i32([w for c in caps for w in c])
        r_feat, r_words = ops.aoa_decoder_lrp(st, self._lrp_weights(), self.num_head, req_img, req_t, req_word,
                                              torch.full_like(req_t, int(head_idx)), tc_gemm=(self.precision in ('bf16', 'mixed')))
        return r_feat, r_words, req_img, req_t, caps

    def explain_caption_words(self, img_filepath):
        """reference :1183-1194: linguistic relevance only (head 0)."""
        self.img_filepath = img_filepath
        self.get_hidden_parameters(img_filepath)
        T = self.caption_length
        _, r_words = self._decoder_lrp(list(range(T)), 0)
        return [r_words[t, :t + 1] for t in range(T)]


# ================================================================================================ gradient family (f4)
from models._gradient import GradientFamily, aoa_grad_weights      # noqa: E402


class ExplainAOAGradient(GradientFamily, ExplainAOAAttention):
    """reference :1257-1592."""
    EX_TYPE = 'gradient'

    def __init__(self, args, word_map, model=None, precision=None):
        ExplainAOAAttention.__init__(self, args, word_map, model=model, precision=precision)
        self._check_encoder()

    def _grad_weights(self):
        return self._cached_grad_weights(aoa_grad_weights)

    def _set_state(self, img, tokens, enc=None):
        ExplainAOAAttention._set_state(self, img, tokens, enc)
        if self._state is not None:
            self.ot_act = self._state["o"][0]

    def gradient_mha(self, d_context, alpha, head_idx):
        """reference :1415-1433: d_value[p, head block] = d_context[head block] * alpha[head, p], zero on the other
        heads.  d_context (1,H) or (H,), alpha (heads,P) -> (P,H).  A tensor expression on the inputs' device; the
        batched path (``lrpx_aoa_decoder_grad_f32``) fuses it."""
        H = self.model.hidden_dim
        dk = H // alpha.size(0)
        d_value = torch.zeros(alpha.size(1), H, device=alpha.device)
        sl = slice(head_idx * dk, (head_idx + 1) * dk)
        d_value[:, sl] = alpha[head_idx].unsqueeze(1) * d_context.reshape(-1)[sl].unsqueeze(0)
        return d_value

    def _decoder_grad(self, ts, head_idx):
        toks = self.beam_caption_encode
        i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=self.device)
        return ops.aoa_decoder_grad(self._state, self._grad_weights(), self.num_head, i32([0] * len(ts)), i32(list(ts)),
                                    i32([toks[t + 1] for t in ts]), i32([head_idx] * len(ts)),
                                    tc_gemm=(self.precision in ('bf16', 'mixed')))

    def explain_caption_wordt(self, t, head_idx):
        """reference :1435-1499 -> (d_img_feature (1,C,h,w), r_words (t+1,))."""
        assert t < self.caption_length
        d_feat, r_words = self._decoder_grad([t], head_idx)
        fh, fw = self._feat_hw
        return d_feat[0].t().reshape(1, -1, fh, fw), r_words[0, :t + 1]

    def explain_caption(self, img_filepath, head_idx, t_list=None):
        """reference :1517-1534."""
        self.img_filepath = img_filepath
        self.get_hidden_parameters(img_filepath)
        if self.caption_length == 0:
            return [], []
        d_feat, r_words = self._decoder_grad(list(range(self.caption_length)), head_idx)
        relevance_imgs, relevance_preceeding_words = self._explain_all(d_feat, r_words)
        self.save_linguistic_explanation(relevance_preceeding_words)
        return relevance_imgs, relevance_preceeding_words

    def explain_caption_words(self, img_filepath, head_idx=0):
        """reference :1536-1548 (whose call omits head_idx and cannot run): linguistic part only."""
        self.img_filepath = img_filepath
        self.get_hidden_parameters(img_filepath)
        _, r_words = self._decoder_grad(list(range(self.caption_length)), head_idx)
        return [r_words[t, :t + 1] for t in range(self.caption_length)]


class ExplainAOAGuidedGradient(ExplainAOAGradient):
    """reference :1594-1666: the decoder half is the plain gradient's, the encoder half guided backpropagation."""
    EX_TYPE = 'GuidedBackpropagate'
    RULE = "guided"


class ExplainAOAGradCam(ExplainAOAGradient):
    """reference :1669-1711."""
    EX_TYPE = 'GradCam'
    CAM = "cam"


class ExplainAOAGuidedGradCam(ExplainAOAGuidedGradient):
    """reference :1714-1776."""
    EX_TYPE = 'GuidedGradCam'
    CAM = "guided"
