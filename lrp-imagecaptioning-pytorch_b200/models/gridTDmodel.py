"""Host-side mirror of the LRP entry points of the reference's models/gridTDmodel.py.

Same class / method names, argument meaning and return values as the reference so that evaluation.py /
train.py style callers can switch over (SURVEY.md §8b):

* ``GridTDModel``  — state_dict-compatible module (reference :106-131) with ``forward`` (:146-198),
  ``beam_search`` (:400-478), and the lrp_tune entry points ``get_lrp_weight_step`` (:549-578),
  ``forwardlrp_context`` (:580-633), ``sample_lrp`` (:635-702).
* ``ExplainGridTDAttention`` — ``get_hidden_parameters`` (:933-1012), ``explain_caption_wordt`` (:1014-1135),
  ``explain_cnn`` (:1137-1139), ``explain_caption`` (:1141-1156), ``teacherforce_forward`` (:892-931),
  ``lrp_linear_eps`` (:744-765).

What differs is HOW the relevance is computed: the per-vector python loops over ``lrp_linear_eps`` become one
batched kernel call per caption (``lrpx_gridtd_decoder_lrp_f32``), the per-sample tuner loop becomes
``lrpx_fc_lrp_weights_f32`` (no ``.item()`` sync), and the encoder relevance runs on the tcgen05 chain
(``lrpx.tc.TcVggEngine``, bf16) or on the fp32 rule kernels through ``LRPtools`` (``precision='fp32'``).
The forward passes that produce the saved state are plain torch tensor ops on the device (library GEMMs).
"""
import os

import torch
import torch.nn as nn

import models.resnet as resnet
import models.vgg as vgg
from LRPtools import lrp_wrapper
from LRPtools import utils as LRPutil
from lrpx import ops
from lrpx import decoder as _dec

try:  # the reference takes nltk's English list (gridTDmodel.py:17-20); fall back to a built-in copy of it
    from nltk.corpus import stopwords as _sw
    STOP_WORDS = list(set(_sw.words('english')))
except Exception:  # pragma: no cover - nltk is not installed in this image
    STOP_WORDS = """i me my myself we our ours ourselves you you're you've you'll you'd your yours yourself yourselves he
    him his himself she she's her hers herself it it's its itself they them their theirs themselves what which who whom
    this that that'll these those am is are was were be been being have has had having do does did doing a an the and
    but if or because as until while of at by for with about against between into through during before after above
    below to from up down in out on off over under again further then once here there when where why how all any both
    each few more most other some such no nor not only own same so than too very s t can will just don don't should
    should've now d ll m o re ve y ain aren aren't couldn couldn't didn didn't doesn doesn't hadn hadn't hasn hasn't
    haven haven't isn isn't ma mightn mightn't mustn mustn't needn needn't shan shan't shouldn shouldn't wasn wasn't
    weren weren't won won't wouldn wouldn't""".split()
STOP_WORDS += ['<start>', '<end>', '<pad>', '<unk>']
BAD_ENDINGS = ['with', 'in', 'on', 'of', 'a', 'at', 'to', 'for', 'an', 'this', 'his', 'her', 'that', 'the', 'and']


class Encoder(nn.Module):
    """reference :23-43"""

    def __init__(self, encoder_type):
        super().__init__()
        if encoder_type == 'resnet101':
            self.encoder = resnet.resnet101(pretrained=True)
            self.feat_dim = self.encoder.feat_dim
        elif encoder_type == 'renset50':          # (sic) the reference's spelling
            self.encoder = resnet.resnet50(pretrained=True)
            self.feat_dim = self.encoder.feat_dim
        elif encoder_type == 'vgg16':
            base_model = vgg.vgg16(pretrained=True)
            self.encoder = base_model.features[0:-1]
            self.feat_dim = base_model.feat_dim
        else:
            raise NotImplementedError("the encoder_type does not exist, please add your encoder_type options")
        self.avgpool = nn.AdaptiveAvgPool2d(1)

    def forward(self, img):
        encoded_image = self.encoder(img)
        return encoded_image, self.avgpool(encoded_image).squeeze()


class AdaptiveLSTMCell(nn.Module):
    """reference :46-58"""

    def __init__(self, input_size, hidden_size):
        super().__init__()
        self.lstm_cell = nn.LSTMCell(input_size, hidden_size)
        self.x_gate = nn.Linear(input_size, hidden_size)
        self.h_gate = nn.Linear(hidden_size, hidden_size)

    def forward(self, inp, states):
        h_old, c_old = states
        ht, ct = self.lstm_cell(inp, (h_old, c_old))
        sen_gate = torch.sigmoid(self.x_gate(inp) + self.h_gate(h_old))
        return ht, ct, sen_gate * torch.tanh(ct)


class AdaptiveAttention(nn.Module):
    """reference :61-103.  The h-projection is broadcast along the *pixel* axis in the image branch (the
    reference's bmm with a ones matrix, :81-87; only shape-valid when the pixel count equals n_pixel, Q19)."""

    def __init__(self, hidden_dim, n_pixel):
        super().__init__()
        self.hidden_dim = hidden_dim
        self.num_pixel = n_pixel
        self.W_v_proj = nn.Linear(hidden_dim, n_pixel)
        self.W_s_proj = nn.Linear(hidden_dim, n_pixel)
        self.W_g_proj = nn.Linear(hidden_dim, n_pixel, bias=False)
        self.w_h = nn.Linear(n_pixel, 1, bias=False)

    def project_image(self, V):
        """V (bs, hidden, P) -> (V^T (bs,P,hidden), W_v V (bs,P,n_pixel)); constant over the time steps."""
        Vt = V.transpose(1, 2)
        return Vt, self.W_v_proj(Vt)

    def attend(self, Vt, img_proj, ht, st):
        ht_proj = self.W_g_proj(ht)                                        # (bs, n_pixel)
        z_t = self.w_h(torch.tanh(img_proj + ht_proj.unsqueeze(2)))        # (bs, P, 1)
        alpha_t = torch.softmax(z_t, dim=1)
        context_t = torch.sum(Vt * alpha_t, dim=1)
        attention_vs = self.w_h(torch.tanh(self.W_s_proj(st) + ht_proj))   # (bs, 1)
        alpha_t_hat = torch.softmax(torch.cat([z_t, attention_vs.unsqueeze(-1)], dim=1), dim=1)
        beta_t = alpha_t_hat[:, -1]                                        # (bs, 1)
        c_t_hat = beta_t * st + (1 - beta_t) * context_t
        return c_t_hat, context_t, alpha_t.squeeze(2), beta_t

    def forward(self, V, ht, st):
        Vt, img_proj = self.project_image(V)
        return self.attend(Vt, img_proj, ht, st)


def _lstm_forward(x, h, c, wi, wh, bi, bh):
    """Hand-rolled LSTM cell returning the pre-tanh candidate and the gate activations (reference :581-592)."""
    z = torch.matmul(x, wi.transpose(0, 1)) + torch.matmul(h, wh.transpose(0, 1)) + bi + bh
    z0, z1, z2, z3 = z.chunk(4, dim=1)
    i = torch.sigmoid(z0)
    f = torch.sigmoid(z1)
    c = f * c + i * torch.tanh(z2)
    h = torch.sigmoid(z3) * torch.tanh(c)
    return h, c, z2, i, f


class GridTDModel(nn.Module):
    """reference :106-702 (the LRP-related surface)."""
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
        self.LanguageLSTM = nn.LSTMCell(2 * hidden_dim, hidden_dim)
        self.AdaLSTM = AdaptiveLSTMCell(embed_dim * 2 + hidden_dim, hidden_dim)
        self.AdaAttention = AdaptiveAttention(self.hidden_dim, n_pixel)
        self.embedding = nn.Embedding(vocab_size, embed_dim)
        self.fc = nn.Linear(hidden_dim, vocab_size)
        self.relu = nn.ReLU()
        self._stop_cache = {}

    # ------------------------------------------------------------------ plain forward / search
    def init_hidden_state(self, V):
        h = torch.zeros(V.shape[0], self.hidden_dim, device=V.device)
        return h, torch.zeros_like(h)

    def predict_next_word(self, image_feature_proj, xt, states):
        h1t, c1t, h2t, c2t = states
        h1t, c1t, st = self.AdaLSTM(xt, (h1t, c1t))
        context_t_hat, context_t, alpha_t, beta_t = self.AdaAttention(image_feature_proj, h1t, st)
        h2t, c2t = self.LanguageLSTM(torch.cat((context_t_hat, h1t), dim=-1), (h2t, c2t))
        predict_score_t = self.fc(self.dropout(context_t_hat + h2t))
        return predict_score_t, alpha_t, beta_t, (h1t, c1t, h2t, c2t)

    def use_tc_encoder(self, precision="fp32"):
        """Frozen VGG encoder ("Training with fixed CNN", train.py:100-104) on the tcgen05 forward: features through
        lrpx.tc.TcVggEngine instead of the library convolutions — 'fp32' = error-compensated bf16x3 (features within
        ~1.5e-4 of the fp32 ones), 'bf16', or None to go back.  Only used while no encoder parameter requires grad."""
        self._tc_encoder_precision = precision
        self._tc_encoder = None

    def _encoder_features(self, images):
        prec = getattr(self, "_tc_encoder_precision", None)
        enc = self.img_encoder.encoder
        if prec and images.is_cuda and isinstance(enc, nn.Sequential) and not any(p.requires_grad for p in enc.parameters()):
            from lrpx import tc
            from LRPtools import lrp_wrapper
            stamp = tuple((p.data_ptr(), p._version) for p in enc.parameters())
            if self._tc_encoder is None or self._tc_encoder[0] != stamp:
                cfgd = lrp_wrapper._tc_cfg(enc)
                if cfgd is None:
                    raise NotImplementedError("use_tc_encoder: the encoder is not a VGG-style conv3x3/ReLU/max-pool stack")
                convs, cfg = cfgd
                if prec == "fp32" and convs[0].out_channels % 64:
                    prec = self._tc_encoder_precision = None          # shapes the general kernels do not take: library forward
                    return self.img_encoder(images)
                # rule='epsilon' keeps ONE accumulator per output channel in the forward (no z+ needed here)
                eng = tc.TcVggEngine([c.weight for c in convs], [c.bias for c in convs], cfg, images.device,
                                     precision="fp32", rule="epsilon") if prec == "fp32" else \
                    tc.TcVggEngine([c.weight for c in convs], [c.bias for c in convs], cfg, images.device)
                self._tc_encoder = (stamp, eng)
            eng = self._tc_encoder[1]
            with torch.no_grad():
                feats = eng.features(eng.forward(images), "nchw")
            return feats, feats.mean((2, 3)).squeeze()
        return self.img_encoder(images)

    def _encode(self, images):
        batch_size = images.size(0)
        image_features, avg_feature = self._encoder_features(images)
        before_act = self.img_projector(image_features)
        image_feature_proj = self.relu(before_act).contiguous().view(batch_size, self.hidden_dim, -1)
        global_before_act = self.global_img_feature_proj(avg_feature)
        global_img_feature = self.relu(global_before_act)
        if global_img_feature.dim() == 1:
            global_img_feature = global_img_feature.unsqueeze(0)
        return image_features, image_feature_proj, global_img_feature

    def forward(self, images, encoded_captions, caption_lengths, ss_prob=None):
        """Teacher-forced forward (reference :146-198; scheduled sampling is not part of the LRP path)."""
        if ss_prob is not None:
            raise NotImplementedError("scheduled sampling is outside the LRP hot path (SURVEY.md §2 #9)")
        batch_size = images.size(0)
        image_features, image_feature_proj, global_img_feature = self._encode(images)
        num_pixels = image_feature_proj.size(-1)
        state = self.init_hidden_state(image_feature_proj) + self.init_hidden_state(image_feature_proj)
        max_length = int(max(caption_lengths)) - 1
        predictions = torch.zeros(batch_size, max_length, self.vocab_size, device=images.device)
        alphas = torch.zeros(batch_size, max_length, num_pixels, device=images.device)
        betas = torch.zeros(batch_size, max_length, 1, device=images.device)
        last_scores = None
        for t in range(max_length):
            word_embedding = self.embedding(encoded_captions[:, t])
            xt = torch.cat((state[2], global_img_feature, word_embedding), dim=-1)
            predict_score_t, alpha_t, beta_t, state = self.predict_next_word(image_feature_proj, xt, state)
            predictions[:, t, :] = predict_score_t
            alphas[:, t, :] = alpha_t
            betas[:, t, :] = beta_t
            last_scores = torch.log_softmax(predict_score_t, -1)
        return predictions, alphas, betas, last_scores, max_length

    def remove_bad_endings(self, sentences):
        """reference :284-300: trailing function words are stripped; a sentence made of nothing else is kept as it
        is (the reference's ``bad_sentence`` branch)."""
        out = []
        for s in sentences:
            words = s.split(' ')
            while words and words[-1] in BAD_ENDINGS:
                words = words[:-1]
            out.append(' '.join(words) if words else s)
        return out

    def beam_search(self, imgs, word_map, beam_size=3, max_cap_length=20):
        """reference :400-478 (batch size 1).  ``beam_idx`` uses floor division — the reference's true division
        (:444) is an IndexError on torch >= 1.6 (Q8)."""
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
            state = self.init_hidden_state(image_feature_proj) + self.init_hidden_state(image_feature_proj)
            unfinished_num = beam_size
            for step in range(max_cap_length):
                word_embedding = self.embedding(k_prev_words).squeeze(1)
                xt = torch.cat((state[2], global_img_feature, word_embedding), dim=-1)
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
            sentence = self.remove_bad_endings([' '.join(rev_word_map[w] for w in sen_idx)])
            return sentence, sen_idx

    def sample(self, images, word_map, caption_lengths, opt={}):
        """reference :200-242 -> (seq, seq_logprobs, max_length): greedy or multinomial sampling without the LRP
        weights (the greedy baseline of the self-critical reward in ``trainciderlrp``, train.py:259-261)."""
        batch_size = images.size(0)
        sample_method = opt.get('sample_method', 'greedy')
        temperature = opt.get('temperature', 1.0)
        max_length = int(max(caption_lengths)) - 1
        _, image_feature_proj, global_img_feature = self._encode(images)
        state = self.init_hidden_state(image_feature_proj) + self.init_hidden_state(image_feature_proj)
        dev = image_feature_proj.device
        seq = torch.zeros(batch_size, max_length, dtype=torch.long, device=dev)
        seq_logprobs = torch.zeros(batch_size, max_length, device=dev)
        it = torch.full((batch_size,), word_map['<start>'], dtype=torch.long, device=dev)
        unfinished = None
        for t in range(max_length):
            xt = torch.cat((state[2], global_img_feature, self.embedding(it)), dim=-1)
            predict_score_t, _, _, state = self.predict_next_word(image_feature_proj, xt, state)
            it, sample_logprobs = self.sample_next_word(torch.log_softmax(predict_score_t, dim=-1), sample_method,
                                                        temperature)
            finished = it == word_map['<end>']
            unfinished = ~finished if unfinished is None else unfinished & ~finished
            it = it * unfinished.type_as(it)
            seq[:, t] = it
            seq_logprobs[:, t] = sample_logprobs.view(-1)
            if int(unfinished.sum()) == 0:
                break
        return seq, seq_logprobs, max_length

    def greedy_search(self, imgs, word_map, max_cap_length=20):
        """reference :480-520 -> (sentences with the bad endings removed, token lists incl. <start>; a finished row
        continues with <pad> = 0).  The BU twin (:2242-2285) is this code over its own ``_encode``."""
        self.eval()
        rev_word_map = {v: k for k, v in word_map.items()}
        with torch.no_grad():
            k_prev_words = torch.zeros(imgs.size(0), max_cap_length, dtype=torch.long, device=imgs.device)
            k_prev_words[:, 0] = word_map['<start>']
            _, image_feature_proj, global_img_feature = self._encode(imgs)
            state = self.init_hidden_state(image_feature_proj) + self.init_hidden_state(image_feature_proj)
            unfinished = None
            for step in range(max_cap_length - 1):
                xt = torch.cat((state[2], global_img_feature, self.embedding(k_prev_words[:, step])), dim=-1)
                predict_score_t, _, _, state = self.predict_next_word(image_feature_proj, xt, state)
                top_words = torch.log_softmax(predict_score_t, dim=-1).topk(1, -1, True, True)[1]
                not_end = top_words != word_map['<end>']
                unfinished = not_end if unfinished is None else unfinished & not_end
                k_prev_words[:, step + 1] = (top_words * unfinished.type_as(top_words))[:, 0]
            seqs = k_prev_words.tolist()
        special = {word_map['<start>'], word_map['<end>'], word_map['<unk>'], word_map['<pad>']}
        sentences = [' '.join(rev_word_map[w] for w in s if w not in special) for s in seqs]
        return self.remove_bad_endings(sentences), seqs

    def beam_search_device(self, imgs, word_map, beam_size=3, max_cap_length=20):
        """``beam_search`` with the whole step loop on the device (lrpx.beam.GridTDBeamSearch: fused step kernels +
        ``lrpx_beam_step`` bookkeeping, one CUDA graph, one read-back) and for B >= 1 images at once.  Same word
        indices as ``beam_search``.  -> (sentence, sen_idx) for one image, a list of such pairs for a batch."""
        from lrpx.beam import GridTDBeamSearch
        self.eval()
        if getattr(self, "_beam", None) is None:
            self._beam = GridTDBeamSearch(self)
        with torch.no_grad():
            _, image_feature_proj, global_img_feature = self._encode(imgs)
        rev_word_map = {v: k for k, v in word_map.items()}
        out = [(self.remove_bad_endings([' '.join(rev_word_map[w] for w in idx)]), idx)
               for idx in self._beam.search(image_feature_proj, global_img_feature, word_map, beam_size, max_cap_length)]
        return out[0] if len(out) == 1 else out

    def sample_next_word(self, logprobs, sample_method, temperature):
        """reference :244-282.  'greedy'; 'gumbel' (arg-max of the Gumbel-perturbed scores, log-probability gathered
        from the unscaled input); anything else samples from softmax(logprobs / temperature) and gathers from the
        SCALED log-probabilities — the reference's top-k / nucleus branch is dead code (`sample_method.startswith ==
        'top'` compares a bound method with a string, :260), so 'top*' behaves like plain sampling there too."""
        if sample_method == 'greedy':
            sampleLogprobs, it = torch.max(logprobs.detach(), 1)
            return it.view(-1).long(), sampleLogprobs
        if sample_method == 'gumbel':
            u = torch.rand(logprobs.shape, device=logprobs.device)
            y = logprobs + (-torch.log(-torch.log(u + 1e-20) + 1e-20))
            it = torch.log_softmax(y / temperature, dim=-1).detach().argmax(1)
            return it, logprobs.gather(1, it.unsqueeze(1))
        logprobs = logprobs / temperature
        it = torch.distributions.Categorical(logits=logprobs.detach()).sample()
        return it, logprobs.gather(1, it.unsqueeze(1))

    # ------------------------------------------------------------------ lrp_tune
    def lrp_linear_eps(self, r_out, forward_input, forward_output, weight):
        """Vector epsilon rule (reference :522-547) on the device: ``lrpx_lrp_linear_eps_f32``.  CUDA tensors only
        (no CPU fallback).  The tuner and the explainer call the batched kernels, which fuse the same arithmetic."""
        return ops.lrp_linear_eps(r_out, forward_input, forward_output, weight)

    def _stop_mask(self, rev_word_map, device):
        key = (id(rev_word_map), str(device))
        m = self._stop_cache.get(key)
        if m is None:
            stop = set(STOP_WORDS)
            m = torch.tensor([rev_word_map.get(i, '<unk>') in stop for i in range(self.vocab_size)],
                             dtype=torch.uint8, device=device)
            self._stop_cache = {key: m}
        return m

    def get_lrp_weight_step(self, predictions_t, rev_word_map, h2t_, context_hat):
        """reference :549-578 — one batched kernel: argmax word (Q16), stop-word skip (Q15), fc epsilon rule,
        split to h2 / context_hat, normalize_relevance (utils.py:55-64).  No host synchronisation."""
        with torch.no_grad():
            w_ctx, w_h, _ = ops.fc_lrp_weights(predictions_t.detach(), h2t_.detach(), context_hat.detach(),
                                               self.fc.weight.detach(), self._stop_mask(rev_word_map, predictions_t.device))
        return w_ctx, w_h

    def _tune_step(self, image_feature_proj, Vt, img_proj, global_img_feature, word_embedding, state):
        x1t_ = torch.cat((state[2], global_img_feature, word_embedding), dim=-1)
        cell = self.AdaLSTM.lstm_cell
        h1_, c1_, _, _, _ = _lstm_forward(x1t_, state[0], state[1], cell.weight_ih, cell.weight_hh, cell.bias_ih,
                                          cell.bias_hh)
        # the tuner takes the sentinel gate from the NEW h1 (reference :617, Q6)
        st_ = torch.sigmoid(self.AdaLSTM.x_gate(x1t_) + self.AdaLSTM.h_gate(h1_)) * torch.tanh(c1_)
        context_t_hat_, _, _, _ = self.AdaAttention.attend(Vt, img_proj, h1_, st_)
        x2t_ = torch.cat((context_t_hat_, h1_), dim=-1)
        L = self.LanguageLSTM
        h2_, c2_, _, _, _ = _lstm_forward(x2t_, state[2], state[3], L.weight_ih, L.weight_hh, L.bias_ih, L.bias_hh)
        return context_t_hat_, (h1_, c1_, h2_, c2_)

    def forwardlrp_context(self, images, encoded_captions, caption_lengths, rev_word_map):
        """reference :580-633 -> (predictions, weighted_predictions, max_length).  Differentiable w.r.t. the
        model parameters; the LRP weights are constants computed under no_grad (:551)."""
        batch_size = images.size(0)
        _, image_feature_proj, global_img_feature = self._encode(images)
        Vt, img_proj = self.AdaAttention.project_image(image_feature_proj)
        state = self.init_hidden_state(image_feature_proj) + self.init_hidden_state(image_feature_proj)
        max_length = int(max(caption_lengths)) - 1
        predictions, weighted = [], []
        for t in range(max_length):
            context_t_hat_, state = self._tune_step(image_feature_proj, Vt, img_proj, global_img_feature,
                                                    self.embedding(encoded_captions[:, t]), state)
            h2_ = state[2]
            predict_score_t = self.fc(context_t_hat_ + h2_)
            weight_context_hat, weight_h2t = self.get_lrp_weight_step(predict_score_t, rev_word_map, h2_, context_t_hat_)
            predictions.append(predict_score_t)
            weighted.append(self.fc(context_t_hat_ * weight_context_hat + weight_h2t * h2_))
        return torch.stack(predictions, 1), torch.stack(weighted, 1), max_length

    def sample_lrp(self, images, rev_word_map, word_map, caption_lengths, opt={}):
        """reference :635-702 -> (seq, seq_logprobs, max_length)."""
        batch_size = images.size(0)
        sample_method = opt.get('sample_method', 'greedy')
        temperature = opt.get('temperature', 1.0)
        max_length = int(max(caption_lengths)) - 1
        _, image_feature_proj, global_img_feature = self._encode(images)
        Vt, img_proj = self.AdaAttention.project_image(image_feature_proj)
        state = self.init_hidden_state(image_feature_proj) + self.init_hidden_state(image_feature_proj)
        dev = images.device
        seq = torch.zeros(batch_size, max_length, dtype=torch.long, device=dev)
        seq_logprobs = torch.zeros(batch_size, max_length, device=dev)
        it = torch.full((batch_size,), word_map['<start>'], dtype=torch.long, device=dev)
        unfinished = None
        for t in range(max_length):
            context_t_hat_, state = self._tune_step(image_feature_proj, Vt, img_proj, global_img_feature,
                                                    self.embedding(it), state)
            h2_ = state[2]
            predict_score_t = self.fc(context_t_hat_ + h2_)
            weight_context_hat, weight_h2t = self.get_lrp_weight_step(predict_score_t, rev_word_map, h2_, context_t_hat_)
            logp = torch.log_softmax(self.fc(context_t_hat_ * weight_context_hat + weight_h2t * h2_), dim=-1)
            it, sample_logprobs = self.sample_next_word(logp, sample_method, temperature)
            finished = it == word_map['<end>']
            unfinished = ~finished if unfinished is None else unfinished & ~finished
            it = it * unfinished.type_as(it)
            seq[:, t] = it
            seq_logprobs[:, t] = sample_logprobs.view(-1)
            if int(unfinished.sum()) == 0:
                break
        return seq, seq_logprobs, max_length


class GridTDModelBU(GridTDModel):
    """reference :1863-2478 — the same decoder on bottom-up region features (B, 36, 2048) instead of images: the
    projector is a ``Linear(2048, hidden)`` over the regions, the global feature is the mean of the PROJECTED regions
    through ``Linear(hidden, embed)`` (:1878-1879, :1911-1916).  ``forward`` / ``beam_search`` / ``get_lrp_weight_step``
    (:2314-2343) / ``forwardlrp_context`` (:2345-2397) / ``sample_lrp`` (:2399-2478) are the parent's code over
    ``_encode``; state_dict keys match the reference's (there is no ``img_encoder``)."""

    def __init__(self, embed_dim, hidden_dim, vocab_size, encoder_type, n_region=36):
        nn.Module.__init__(self)
        self.embed_dim = embed_dim
        self.hidden_dim = hidden_dim
        self.vocab_size = vocab_size
        self.encoder_type = encoder_type
        self.dropout = nn.Dropout(0.5)
        self.encoder_raw_dim = 2048
        self.img_projector = nn.Linear(self.encoder_raw_dim, self.hidden_dim)
        self.global_img_feature_proj = nn.Linear(self.hidden_dim, self.embed_dim)
        self.LanguageLSTM = nn.LSTMCell(2 * hidden_dim, hidden_dim)
        self.AdaLSTM = AdaptiveLSTMCell(embed_dim * 2 + hidden_dim, hidden_dim)
        self.AdaAttention = AdaptiveAttention(self.hidden_dim, n_region)
        self.embedding = nn.Embedding(vocab_size, embed_dim)
        self.fc = nn.Linear(hidden_dim, vocab_size)
        self.relu = nn.ReLU()
        self._stop_cache = {}

    def _encode(self, images_features):
        proj = self.relu(self.img_projector(images_features))                 # (bs, regions, hidden)
        global_img_feature = self.relu(self.global_img_feature_proj(torch.mean(proj, dim=1)))
        if global_img_feature.dim() == 1:
            global_img_feature = global_img_feature.unsqueeze(0)
        return images_features, proj.contiguous().transpose(1, 2), global_img_feature     # (bs, hidden, regions)


# ----------------------------------------------------------------------------------------------------
class ExplainGridTDAttention(object):
    """reference :705-1211.  ``precision`` (a keyword the reference does not have; default 'fp32'):
      'fp32' — the reference's fp32 bar.  VGG encoders: the tcgen05 chain in its fp32-accurate mode (error-compensated
               bf16x3 operands, fp32 gains, hi|lo inter-layer storage); other encoders: the fp32 CUDA-core rule kernels
               through LRPtools.  Decoder GEMMs on fp32 CUDA cores.
      'bf16' — VGG encoders only: the tcgen05 chain with bf16 operands / storage (Spearman >= 0.99, rel-L2 <= 5e-2 vs
               the reference), decoder GEMMs as bf16x3 on tensor cores.  The throughput mode of bench.py.
      'mixed' — VGG encoders: the encoder FORWARD in the fp32-accurate mode (once per image), the relevance chain in
               bf16 (lrpx.tc.TcVggMixed): accurate features for the decoder and accurate max-pool winners at ~0.85 of
               the bf16 mode's throughput.
      'simt' — the fp32 CUDA-core rule kernels through LRPtools whatever the encoder."""
    EPS = LRPutil.EPSILON
    EX_TYPE = 'lrp'
    # the reference never zeroes sample.grad, so relevance_imgs[t] of explain_caption is the running sum over
    # the words explained so far (Q1); set False for per-word heat-maps
    ACCUMULATE_LIKE_REFERENCE = True

    def __init__(self, args, word_map, model=None, precision=None):
        self._common_init(args, word_map, model, precision,
                          lambda: GridTDModel(args.embed_dim, args.hidden_dim, len(word_map), args.encoder))
        m = self.model
        self.adalstm_weight_i, self.adalstm_weight_h = m.AdaLSTM.lstm_cell.weight_ih, m.AdaLSTM.lstm_cell.weight_hh
        self.adalstm_bias_i, self.adalstm_bias_h = m.AdaLSTM.lstm_cell.bias_ih, m.AdaLSTM.lstm_cell.bias_hh

    def _common_init(self, args, word_map, model, precision, make_model):
        self.args = args
        self.word_map = word_map
        self.vocab_size = len(word_map)
        if model is not None:
            self.model = model
        else:
            self.model = make_model()
            checkpoint = torch.load(args.weight, map_location='cpu')
            self.model.load_state_dict(checkpoint['state_dict'])
            self.model.cuda()
        self.model.eval()
        # the forward passes are torch tensor ops; every relevance call below goes to liblrpx.so, which raises
        # on non-CUDA tensors (there is no CPU fallback)
        self.device = next(self.model.parameters()).device
        # bottom-up twins (GridTDModelBU / AOAModelBU) have no CNN: the explanation ends at the region features
        self.has_encoder = hasattr(self.model, 'img_encoder')
        is_vgg = self.has_encoder and isinstance(self.model.img_encoder.encoder, nn.Sequential)
        self.precision = precision or 'fp32'
        if self.precision not in ('fp32', 'bf16', 'simt', 'mixed'):
            raise ValueError(f"precision must be 'fp32', 'bf16', 'mixed' or 'simt', got {self.precision!r}")
        tcp = lrp_wrapper._tc_cfg(self.model.img_encoder.encoder) if is_vgg else None
        # the general kernels (fp32-accurate mode) need a first conv with a multiple of 64 output channels
        tc_ok = tcp is not None and (self.precision == 'bf16' or tcp[0][0].out_channels % 64 == 0)
        # Bottleneck ResNets run the bf16 chain of lrpx.tc_resnet (their fp32 bar is the CUDA-core rule path)
        self.is_resnet = self.has_encoder and lrp_wrapper._is_bottleneck_resnet(self.model.img_encoder.encoder)
        if self.is_resnet and self.precision == 'bf16':
            tc_ok = True
        if self.precision == 'bf16' and not tc_ok and self.has_encoder:
            raise NotImplementedError("the tensor-core chain supports VGG-style encoders; use precision='fp32'")
        # the encoder runs on the tcgen05 engine (one forward per image shared by all its words)
        if self.precision == 'mixed' and not (tc_ok and not self.is_resnet):
            raise NotImplementedError("precision='mixed' needs a VGG-style encoder with a 64-channel first layer")
        self.uses_tc = tc_ok and self.precision in ('fp32', 'bf16', 'mixed')
        self.mean = [0.485, 0.456, 0.406]
        self.std = [0.229, 0.224, 0.225]
        m = self.model
        if hasattr(m, 'LanguageLSTM'):       # the single-LSTM adaptive attention model has none
            self.language_weight_i, self.language_weight_h = m.LanguageLSTM.weight_ih, m.LanguageLSTM.weight_hh
            self.language_bias_i, self.language_bias_h = m.LanguageLSTM.bias_ih, m.LanguageLSTM.bias_hh
        self.output_weight = m.fc.weight
        self.visualizatioin_save_path = os.path.join(args.save_path, args.dataset + 'explanation')
        os.makedirs(self.visualizatioin_save_path, exist_ok=True)
        self._engine = self._engine_key = None
        self._weights = self._weights_key = None
        self._state = None

    # ------------------------------------------------------------------ helpers
    def lrp_linear_eps(self, r_out, forward_input, forward_output, weight):
        """reference :744-765 on the device: ``lrpx_lrp_linear_eps_f32`` (CUDA tensors only, no CPU fallback)."""
        return ops.lrp_linear_eps(r_out, forward_input, forward_output, weight)

    def preprocess_img(self, img_filepath):
        """reference :767-771: Resize((height,width)) -> ToTensor -> Normalize."""
        from PIL import Image
        import numpy as np
        img = Image.open(img_filepath).convert('RGB').resize((self.args.width, self.args.height), Image.BILINEAR)
        x = torch.from_numpy(np.asarray(img, dtype=np.float32) / 255.).permute(2, 0, 1)
        x = (x - torch.tensor(self.mean).view(3, 1, 1)) / torch.tensor(self.std).view(3, 1, 1)
        return x.unsqueeze(0).to(self.device)

    def _lrp_weights(self):
        """The decoder relevance kernels' weights (gate rows concatenated, projector reshaped), rebuilt when a model
        parameter is replaced or updated in place; the dict stays the same object until then."""
        key = ops.weight_stamp(self.model.parameters())
        if self._weights is None or self._weights_key != key:
            sd = {k: v.detach() for k, v in self.model.state_dict().items()}
            self._weights, self._weights_key = _dec.gridtd_weights(sd), key
        return self._weights

    def _encoder_stamp(self):
        enc = getattr(getattr(self.model, "img_encoder", None), "encoder", None)
        return () if enc is None else ops.weight_stamp(list(enc.parameters()) + list(enc.buffers()))

    def engine(self):
        """The tensor-core encoder engine (it holds converted copies of the encoder's weights): rebuilt when an encoder
        parameter or buffer changes."""
        key = self._encoder_stamp()
        if self._engine is not None and self._engine_key != key:
            self._engine = None
        self._engine_key = key
        if self._engine is None and getattr(self, "is_resnet", False):
            from lrpx import tc_resnet
            self._engine = tc_resnet.TcResNetEngine(self.model.img_encoder.encoder, self.device)
        if self._engine is None:
            from lrpx import tc
            enc = self.model.img_encoder.encoder
            convs = [m for m in enc if isinstance(m, nn.Conv2d)]
            cfg = []
            for m in enc:
                if isinstance(m, nn.Conv2d):
                    cfg.append(m.out_channels)
                elif isinstance(m, nn.MaxPool2d):
                    cfg.append("M")
            if self.precision == 'mixed':
                self._engine = tc.TcVggMixed([c.weight for c in convs], [c.bias for c in convs], cfg, self.device)
            else:
                self._engine = tc.TcVggEngine([c.weight for c in convs], [c.bias for c in convs], cfg, self.device,
                                              precision=self.precision)
        return self._engine

    def encode_images(self, imgs):
        """Encoder forward -> (features (B,P,C) fp32 pixel-major, feature map size, encoder state)."""
        if self.uses_tc:
            eng = self.engine()
            est = eng.forward(imgs)
            return eng.features(est, "pixel"), est.feat_hw, est
        enc = self.model.img_encoder.encoder
        if not hasattr(enc, "_lrpx_plan"):
            lrp_wrapper.add_lrp(enc)
        with torch.no_grad():
            fmap = enc._lrpx_plan.forward(imgs.detach().float())
        B, C, h, w = fmap.shape
        return fmap.flatten(2).transpose(1, 2).contiguous(), (h, w), None

    def _explainer_weights(self, quirk_double_bias_ih=True):
        """Concatenated / re-laid-out weights of the fused explainer forward, cached until a parameter changes
        (the cache key holds every source tensor's data pointer and in-place version counter)."""
        m = self.model
        cell, L, xg, hg = m.AdaLSTM.lstm_cell, m.LanguageLSTM, m.AdaLSTM.x_gate, m.AdaLSTM.h_gate
        src = [cell.weight_ih, cell.weight_hh, cell.bias_ih, cell.bias_hh, xg.weight, xg.bias, hg.weight, hg.bias,
               L.weight_ih, L.weight_hh, L.bias_ih, L.bias_hh]
        key = (quirk_double_bias_ih,) + tuple((t.data_ptr(), t._version) for t in src)
        if getattr(self, "_expl_w_key", None) != key:
            H = m.hidden_dim
            with torch.no_grad():
                # x1 = [h2, glob, emb] (:975): recurrent part [h2 | h1] -> (4H gates | sentinel gate), input part [glob | emb]
                W1_rec = torch.cat((torch.cat((cell.weight_ih[:, :H], cell.weight_hh), 1),
                                    torch.cat((xg.weight[:, :H], hg.weight), 1)), 0).t().contiguous()      # (2H, 5H)
                W1_in = torch.cat((cell.weight_ih[:, H:], xg.weight[:, H:]), 0).t().contiguous()           # (2E, 5H)
                b1 = torch.cat((cell.bias_ih + cell.bias_hh, xg.bias + hg.bias)).contiguous()
                W2 = torch.cat((L.weight_ih, L.weight_hh), 1).t().contiguous()                             # (3H, 4H)
                b2 = (L.bias_ih + (L.bias_ih if quirk_double_bias_ih else L.bias_hh)).contiguous()        # Q3 (:789)
                self._expl_w = (ops.lstm_prep_weights(W1_rec, 5), W1_in, b1, ops.lstm_prep_weights(W2, 4), b2)
            self._expl_w_key = key
        return self._expl_w

    def _lx(self, name, weight, bias=None, derive=None):
        """Cached tensor-core Linear for the explainer forwards: ``weight`` (out, in) and ``bias`` are (views of) model
        parameters; ``derive()`` (optional) builds the actual (weight, bias) from them (concatenations, transposes) and
        is re-run only when a source tensor changes (data pointer / in-place version)."""
        src = [t for t in (weight if isinstance(weight, (list, tuple)) else [weight]) if t is not None]
        src += [t for t in (bias if isinstance(bias, (list, tuple)) else [bias]) if t is not None]
        key = tuple((t.data_ptr(), t._version) for t in src)
        cache = self.__dict__.setdefault("_lx_cache", {})
        hit = cache.get(name)
        if hit is None or hit[0] != key:
            with torch.no_grad():
                w, b = derive() if derive is not None else (weight.detach(), None if bias is None else bias.detach())
            hit = cache[name] = (key, self._linear(w, b), (w, b))
        return hit[1]

    def _linear(self, weight, bias):
        """A Linear layer of the explainer forward.  precision 'bf16' (the throughput mode): ``ops.LinearX3`` — the
        tcgen05 GEMM with error-compensated bf16x3 operands (measured 2-3e-6 of sum |x w| off fp64, one-sided by the
        tensor cores' round-toward-zero accumulation) — for the shapes it takes.  'fp32' / 'simt' keep the fp32 library
        GEMM: their bar is the reference's elementwise rtol 1e-4 / atol 1e-6 on the saved state."""
        if self.precision in ('bf16', 'mixed') and ops.LinearX3.supports(weight):
            return ops.LinearX3(weight, bias)
        return lambda x: torch.addmm(bias, x, weight.t()) if bias is not None else x @ weight.t()

    def _linears(self):
        """The explainer forward's Linear layers on the tensor-core GEMM (built once, rebuilt when a source parameter
        changes): 1x1 projector, global projection, W_v, the input-side gate pre-activations, the two attention
        projections as one block-diagonal layer, the vocabulary projection."""
        m = self.model
        att, cell, xg = m.AdaAttention, m.AdaLSTM.lstm_cell, m.AdaLSTM.x_gate
        src = [m.img_projector.weight, m.img_projector.bias, m.global_img_feature_proj.weight, att.W_v_proj.weight,
               att.W_g_proj.weight, att.W_s_proj.weight, att.W_s_proj.bias, m.fc.weight, m.fc.bias, cell.weight_ih,
               cell.bias_ih, cell.bias_hh, xg.weight, xg.bias]
        key = tuple((t.data_ptr(), t._version) for t in src)
        if getattr(self, "_lin_key", None) != key:
            H, K = m.hidden_dim, att.num_pixel
            dev = m.fc.weight.device
            _, W1_in, b1, _, _ = self._explainer_weights()
            with torch.no_grad():
                Wa = torch.zeros(2 * K, 2 * H, device=dev)                 # (out, in): rows 0..K-1 <- h1, K..2K-1 <- s
                Wa[:K, :H] = att.W_g_proj.weight
                Wa[K:, H:] = att.W_s_proj.weight
                ba = torch.cat((torch.zeros(K, device=dev), att.W_s_proj.bias))
                Wp = m.img_projector.weight.detach().reshape(H, -1)
                W1t = W1_in.t().contiguous()
            L = self._linear
            self._lin = dict(proj=L(Wp, m.img_projector.bias.detach()),
                             glob=L(m.global_img_feature_proj.weight.detach(), m.global_img_feature_proj.bias.detach()),
                             wv=L(att.W_v_proj.weight.detach(), att.W_v_proj.bias.detach()), pre1=L(W1t, b1), att=L(Wa, ba),
                             fc=L(m.fc.weight.detach(), m.fc.bias.detach()))
            self._lin_key = key
        return self._lin

    def explainer_forward(self, feat, tokens, quirk_double_bias_ih=True, want_gates=False):
        """The explainer's teacher-forced forward (reference :941-1012) batched over images.

        feat: (B,P,C) pixel-major encoder output; tokens: (B,L) long, column 0 = <start>.  Returns the saved
        state in the kernels' layout (lrpx_gridtd_args), T = L-1 steps.  ``quirk_double_bias_ih`` reproduces the
        explainer's language LSTM adding bias_ih twice (:789, Q3).

        A time step is three kernels writing straight into the saved-state tensors: ``lrpx_lstm_step_f32`` (skinny
        GEMM over the concatenated recurrent inputs + cell rule) for the AdaLSTM, ``lrpx_adaptive_attention_f32``
        (both attention projections + attention + sentinel mix), ``lrpx_lstm_step_f32`` for the language LSTM;
        everything that does not depend on the recurrent state (embeddings, the input-side halves of the gate
        pre-activations, the vocabulary projection) is one batched GEMM over all T steps.  CUDA only: there is no
        CPU form in the product (tests/helpers.py holds the step-by-step tensor-op restatement the kernels are
        checked against).  ``want_gates`` also saves the output gates and the sentinel gate (o1, o2, sg): the state
        of the gradient explainers (reference :1381-1419)."""
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
        lin = self._linears()         # the forward's GEMMs on the tcgen05 kernels (bf16x3: fp32 accuracy), no library GEMM
        with torch.no_grad():
            feat = feat.contiguous()
            avg = feat.mean(1)
            A_pre = lin["proj"](feat.view(B * P, C)).view(B, P, H)
            A = A_pre.clamp(min=0)
            glob_pre = lin["glob"](avg)
            glob = glob_pre.clamp(min=0)
            img_proj = lin["wv"](A.view(B * P, H)).view(B, P, K)                     # (B,P,K)
            cell, L = m.AdaLSTM.lstm_cell, m.LanguageLSTM
            W1p, W1_in, b1, W2p, b2 = self._explainer_weights(quirk_double_bias_ih)
            # both attention projections as ONE GEMM per step: [h1 | s] @ blockdiag(W_g^T, W_s^T) + [0 | b_s]
            # (computing them inside the attention kernel re-reads 0.8 MB of weights per image and step: measured slower)
            w_h = att.w_h.weight.reshape(-1).contiguous()
            # ---- state-independent halves for all T steps at once
            emb = m.embedding(tokens[:, :T])                                                     # (B,T,E)
            xin = torch.cat((glob.unsqueeze(1).expand(B, T, E), emb), -1)                        # (B,T,2E)
            pre1 = lin["pre1"](xin.transpose(0, 1).reshape(T * B, 2 * E)).view(T, B, 5 * H)
            # ---- saved state
            h1, c1, h2, c2 = (torch.zeros(B, T + 1, H, device=dev) for _ in range(4))
            g1, i1, f1, g2, i2, f2, st, ctx, ctx_hat = (new(B, T, H) for _ in range(9))
            alpha, beta = new(B, T, P), new(B, T)
            o1, o2, sg = (new(B, T, H) for _ in range(3)) if want_gates else (None, None, None)
            row = lambda x, t: None if x is None else x[:, t]
            # ---- staging rows of the recurrent GEMMs, ping-ponged over the steps: a step kernel reads ALL columns of
            # its input rows in every CTA while its CTAs write the new state, so the new state goes to the other copy
            hcat = torch.zeros(2, B, 2 * H, device=dev)       # [h2_t | h1_t]
            x2c = torch.zeros(2, B, 3 * H, device=dev)        # [ctx_hat_t | h1_{t+1} | h2_t]
            hs = new(B, 2 * H)                                # [h1_{t+1} | s_t]
            for t in range(T):
                p, q = t & 1, (t & 1) ^ 1
                # AdaLSTM: 4 gates + sentinel gate from [h2_t | h1_t] (+ the input-side halves in pre1[t])   :975-983
                ops.lstm_step(hcat[p], W1p, pre1[t], 5, c1[:, t], h1[:, t + 1], c1[:, t + 1], g1[:, t], i1[:, t],
                              f1[:, t], s=st[:, t], h_copy0=hcat[q][:, H:], h_copy1=x2c[p][:, H:2 * H],
                              h_copy2=hs[:, :H], s_copy=hs[:, H:], o=row(o1, t), sg=row(sg, t))
                hsp = lin["att"](hs)                                                              # (B,2K)
                ops.adaptive_attention(A, img_proj, hsp, w_h, st[:, t], ctx[:, t], ctx_hat[:, t], alpha[:, t],
                                       beta[:, t], ctx_hat_copy=x2c[p][:, :H])
                # LanguageLSTM from [ctx_hat_t | h1_{t+1} | h2_t]                                             :984-990
                ops.lstm_step(x2c[p], W2p, b2, 4, c2[:, t], h2[:, t + 1], c2[:, t + 1], g2[:, t], i2[:, t], f2[:, t],
                              h_copy0=hcat[q][:, :H], h_copy1=x2c[q][:, 2 * H:], o=row(o2, t))
            pred = lin["fc"]((ctx_hat + h2[:, 1:]).view(B * T, H)).view(B, T, m.vocab_size)
            x1 = torch.cat((h2[:, :T], xin), -1)
            x2 = torch.cat((ctx_hat, h1[:, 1:]), -1)
            st_ = dict(x1=x1, x2=x2, g1=g1, i1=i1, f1=f1, g2=g2, i2=i2, f2=f2, st=st, ctx=ctx, ctx_hat=ctx_hat,
                       alpha=alpha, beta=beta, pred=pred, h1=h1, c1=c1, h2=h2, c2=c2, feat=feat, avg=avg,
                       A_pre=A_pre.contiguous(), A=A.contiguous(), glob_pre=glob_pre)
            if want_gates:
                st_.update(o1=o1, o2=o2, sg=sg)
        return st_

    def teacherforce_forward(self, img, beam_caption_encode):
        """reference :892-931 -> logits (len(beam_caption_encode), vocab)."""
        feat, _, _ = self.encode_images(img)
        toks = torch.tensor([list(beam_caption_encode) + [0]], dtype=torch.long, device=self.device)
        return self.explainer_forward(feat, toks)["pred"][0]

    # ------------------------------------------------------------------ reference entry points
    # with the tensor-core encoder the caption search runs on the device too and shares the encoder pass of the
    # explanation (the reference's host loop encodes the image a second time); set False for the host loop
    DEVICE_BEAM_SEARCH = True
    _BEAM = "GridTDBeamSearch"            # class in lrpx.beam
    _REMOVE_BAD_ENDINGS = True

    def _search_inputs(self, feat):
        """(B,P,C) encoder features -> what the model's ``_encode`` hands to its beam search."""
        m = self.model
        B, P, C = feat.shape
        Wp = m.img_projector.weight.reshape(m.hidden_dim, -1)
        proj = torch.addmm(m.img_projector.bias, feat.reshape(B * P, C), Wp.t()).clamp(min=0).view(B, P, -1)
        return proj.transpose(1, 2), m.global_img_feature_proj(feat.mean(1)).clamp(min=0)           # (B,H,P), (B,E)

    def _find_caption(self, img_filepath, beam_size, max_cap_length):
        """Sets ``beam_caption`` / ``beam_caption_encode`` (with <start>) from the model's beam search; returns the
        encoder pass when it was already needed for the search (device search), else None."""
        m = self.model
        enc = None
        if (self.DEVICE_BEAM_SEARCH and self.uses_tc and self.has_encoder and self.img.is_cuda
                and 'beam_search' not in m.__dict__):
            from lrpx import beam
            if getattr(self, "_beam", None) is None:
                self._beam = getattr(beam, self._BEAM)(m)
            enc = self.encode_images(self.img)
            with torch.no_grad():
                proj, glob = self._search_inputs(enc[0])
            idx = self._beam.search(proj, glob, self.word_map, beam_size=beam_size, max_cap_length=max_cap_length)[0]
            if getattr(self, "_rev_word_map", None) is None:          # built once: ~1 ms for a 10 000-word vocabulary
                self._rev_word_map = {v: k for k, v in self.word_map.items()}
            rev = self._rev_word_map
            sentence = [' '.join(rev[w] for w in idx)]
            self.beam_caption = m.remove_bad_endings(sentence) if self._REMOVE_BAD_ENDINGS else sentence
            self.beam_caption_encode = idx
        else:
            self.beam_caption, self.beam_caption_encode = m.beam_search(self.img, self.word_map, beam_size=beam_size,
                                                                        max_cap_length=max_cap_length)
        self.beam_caption_encode = [self.word_map['<start>']] + self.beam_caption_encode
        print(f'the predicted caption of {img_filepath} is "{self.beam_caption[0]}"')
        return enc

    def get_hidden_parameters(self, img_filepath):
        self.img = self.preprocess_img(img_filepath)
        enc = self._find_caption(img_filepath, beam_size=2, max_cap_length=50)
        self._set_state(self.img, self.beam_caption_encode, enc)

    def forward_greedy(self, img_filepath):
        """reference :799-890: the saved state for the beam-size-1 caption of at most 20 words."""
        self.img = self.preprocess_img(img_filepath)
        enc = self._find_caption(img_filepath, beam_size=1, max_cap_length=20)
        self._set_state(self.img, self.beam_caption_encode, enc)

    def _empty_caption(self, tokens):
        """The search returned no word (<end> or only special tokens first): like the reference, nothing is explained
        (caption_length 0, explain_caption returns two empty lists)."""
        if len(tokens) > 1:
            return False
        self._state, self._enc_state, self.caption_length = None, None, 0
        self.predictions = torch.zeros(0, self.vocab_size, device=self.device)
        return True

    def _set_state(self, img, tokens, enc=None):
        if self._empty_caption(tokens):
            return
        feat, (fh, fw), est = enc if enc is not None else self.encode_images(img)
        toks = torch.tensor([tokens], dtype=torch.long, device=self.device)
        st = self.explainer_forward(feat, toks)
        self._state, self._enc_state, self._feat_hw = st, est, (fh, fw)
        self.caption_length = len(tokens) - 1
        self.num_pixels = feat.shape[1]
        # attributes the reference exposes (read by evaluation.py: .predictions .alphas .betas ...)
        self.predictions, self.alphas, self.betas = st["pred"][0], st["alpha"][0], st["beta"][0]
        self.x1t, self.x2t = st["x1"][0], st["x2"][0]
        self.h1t, self.c1t, self.h2t, self.c2t = st["h1"][0], st["c1"][0], st["h2"][0], st["c2"][0]
        self.g1t, self.i1t_act, self.f1t_act = st["g1"][0], st["i1"][0], st["f1"][0]
        self.g2t, self.i2t_act, self.f2t_act = st["g2"][0], st["i2"][0], st["f2"][0]
        self.st, self.context, self.context_hat = st["st"][0], st["ctx"][0], st["ctx_hat"][0]
        C = feat.shape[2]
        self.image_features = feat[0].t().reshape(1, C, fh, fw)
        self.avg_feature = st["avg"][0]

    def _decoder_lrp(self, ts):
        toks = self.beam_caption_encode
        dev = self.device
        req_t = torch.tensor(ts, dtype=torch.int32, device=dev)
        req_word = torch.tensor([toks[t + 1] for t in ts], dtype=torch.int32, device=dev)
        req_img = torch.zeros(len(ts), dtype=torch.int32, device=dev)
        return ops.gridtd_decoder_lrp(self._state, self._lrp_weights(), req_img, req_t, req_word,
                                      tc_gemm=(self.precision in ('bf16', 'mixed')))

    def explain_caption_wordt(self, t):
        """reference :1014-1135 -> (r_img_feature (1,C,h,w), r_words (t+1,))."""
        assert t < self.caption_length
        r_feat, r_words = self._decoder_lrp([t])
        fh, fw = self._feat_hw
        r_img_feature = r_feat[0].t().reshape(1, -1, fh, fw)
        return r_img_feature, r_words[0, :t + 1]

    def explain_cnn(self, r_img_feature):
        """reference :1137-1139: relevance of the encoder output -> relevance of the image (1,3,H,W)."""
        if self.uses_tc:
            r_pix = r_img_feature.flatten(2).transpose(1, 2).contiguous()
            return self.engine().relevance(self._enc_state, r_pix)
        enc = self.model.img_encoder.encoder
        if not hasattr(enc, "_lrpx_plan"):
            lrp_wrapper.add_lrp(enc)
        return enc.compute_lrp(self.img, target=r_img_feature, precision='simt')

    def explain_caption(self, img_filepath, t_list=None):
        """reference :1141-1156 -> (relevance_imgs [T x (1,3,H,W)], relevance_preceeding_words [T x (t+1,)]).
        All words of the caption are explained in one batched decoder call + one batched encoder chain."""
        self.img_filepath = img_filepath
        self.get_hidden_parameters(img_filepath)
        T = self.caption_length
        if T == 0:
            return [], []
        r_feat, r_words = self._decoder_lrp(list(range(T)))
        if self.uses_tc:
            rows = torch.zeros(T, dtype=torch.int32, device=self.device)
            heat = self.engine().relevance(self._enc_state, r_feat, rows)
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
        self.visualize_explanations(relevance_imgs, t=t_list)
        self.save_linguistic_explanation(relevance_preceeding_words)
        return relevance_imgs, relevance_preceeding_words

    def save_linguistic_explanation(self, relevance_preceeding_words):
        """reference :1158-1174 (yaml dump of the per-word relevances)."""
        import yaml
        name = os.path.basename(self.img_filepath)
        save_dir = os.path.join(self.visualizatioin_save_path, name[:-4] if name.endswith('.jpg') else name)
        os.makedirs(save_dir, exist_ok=True)
        words = ['<start>'] + self.beam_caption[0].split(' ')
        out = []
        for t in range(min(self.caption_length, len(words) - 1)):
            rel = relevance_preceeding_words[t].tolist()
            out.append({words[t + 1]: [{words[i]: rel[i]} for i in range(len(rel))]})
        with open(os.path.join(save_dir, self.EX_TYPE + '_linguistic_explanation.yaml'), 'w') as f:
            yaml.safe_dump(out, f)

    def visualize_explanations(self, relevance_imgs, t=None):
        """The reference renders matplotlib figures (:1176-1211); plotting is out of scope (SURVEY.md §2 #3)."""
        return None


# ================================================================================================ gradient family (f4)
from models._gradient import GradientFamily, gridtd_grad_weights      # noqa: E402  (after the classes it extends)


class ExplainGridTDGradient(GradientFamily, ExplainGridTDAttention):
    """reference :1214-1582.  Gradient of the target word's logit with respect to the image (the decoder's attention
    weights and gates held constant, as the reference's hand-written backward does) and the per-word sums of the
    embedding gradients.  ``model=`` / ``precision=`` are keywords the reference does not have."""
    EX_TYPE = 'gradient'

    def __init__(self, args, word_map, model=None, precision=None):
        ExplainGridTDAttention.__init__(self, args, word_map, model=model, precision=precision)
        self._check_encoder()

    def _grad_weights(self):
        return self._cached_grad_weights(gridtd_grad_weights)

    def get_hidden_parameters(self, img_filepath):
        """reference :1323-1422 (beam size 3, up to 50 words)."""
        self.img = self.preprocess_img(img_filepath)
        enc = self._find_caption(img_filepath, beam_size=3, max_cap_length=50)
        self._set_state(self.img, self.beam_caption_encode, enc)

    def _set_state(self, img, tokens, enc=None):
        ExplainGridTDAttention._set_state(self, img, tokens, enc)
        if self._state is not None:
            st = self._state
            self.o1t_act, self.o2t_act, self.sen_gate = st["o1"][0], st["o2"][0], st["sg"][0]

    def _decoder_grad(self, ts):
        toks = self.beam_caption_encode
        i32 = lambda v: torch.tensor(v, dtype=torch.int32, device=self.device)
        return ops.gridtd_decoder_grad(self._state, self._grad_weights(), i32([0] * len(ts)), i32(list(ts)),
                                       i32([toks[t + 1] for t in ts]), guided=self.GUIDED_DECODER,
                                       tc_gemm=(self.precision in ('bf16', 'mixed')))

    def explain_caption_wordt(self, t):
        """reference :1424-1508 (guided: :1588-1675) -> (d_img_feature (1,C,h,w), r_words (t+1,))."""
        assert t < self.caption_length
        d_feat, r_words = self._decoder_grad([t])
        fh, fw = self._feat_hw
        return d_feat[0].t().reshape(1, -1, fh, fw), r_words[0, :t + 1]

    def explain_caption(self, img_filepath, t_list=None):
        """reference :1525-1539: every word of the caption in one batched decoder call + one batched encoder pass."""
        self.img_filepath = img_filepath
        self.get_hidden_parameters(img_filepath)
        if self.caption_length == 0:
            return [], []
        d_feat, r_words = self._decoder_grad(list(range(self.caption_length)))
        return self._explain_all(d_feat, r_words)


class ExplainiGridTDGuidedGradient(ExplainGridTDGradient):
    """reference :1585-1749 (the class name's typo is the reference's): guided backpropagation."""
    EX_TYPE = 'GuidedBackpropagate'
    RULE = "guided"
    GUIDED_DECODER = True


class ExplainGridTDGradCam(ExplainGridTDGradient):
    """reference :1752-1793: explain_cnn returns the (1, P) Grad-CAM map of the encoder output."""
    EX_TYPE = 'GradCam'
    CAM = "cam"


class ExplainGridTDGuidedGradCam(ExplainiGridTDGuidedGradient):
    """reference :1796-1859: guided backpropagation times the pyramid-expanded Grad-CAM map."""
    EX_TYPE = 'GuidedGradCam'
    CAM = "guided"
