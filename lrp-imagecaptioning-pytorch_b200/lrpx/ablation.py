"""Ablation experiments of the reference's evaluation.py (SURVEY.md §8 f3), batched over (image, word) requests.

``EvaluationExperiments.ablation_experiment`` (evaluation.py:82-290) walks one image at a time and, per explained word,

* image ablation (:120-150): blanks the 20 most relevant 8x8 patches of the image (``block_image`` :57-80), captions
  the modified image again with beam search, and records whether the word disappears or — if it is still there — how
  much its softmax score drops under teacher forcing of the new prefix;
* word ablation (:234-262): deletes the 3 most relevant preceding words and records the score drop of the word under
  teacher forcing of the shortened prefix.

Here every stage runs once for ALL requests: ``lrpx_block_image_f32`` writes the masked images, the tensor-core encoder
and the device beam search (lrpx.beam) caption them in chunks, and one batched explainer forward per experiment yields
the teacher-forced scores; ``lrpx_bbox_ratio_f32`` scores every heat-map against its bounding boxes
(``bbox_experiment``, :344-447).  The word filters of the reference (object-word list, stop words, t >= 1 / t >= 6) are the
caller's choice of requests.
"""
import torch

from . import ops


class AblationExperiments:
    def __init__(self, explainer, num_delete_patches=20, patch_size=8, num_delete_words=3, chunk=128):
        """explainer: ExplainGridTDAttention / ExplainAOAAttention / ExplainAdaptiveAttention with precision='bf16'
        (VGG encoder on the tensor-core engine).  Defaults: evaluation.py:55-56, :241.
        The heat-maps come from the caller, typically ``lrpx.pipeline.BatchExplainer(...).explain`` or ``explain_images``
        of any image-resolution method: LRP, the gradient, guided backpropagation or Guided Grad-CAM (its maps have the
        same (Q,3,H,W) shape and delivery formats).  Grad-CAM's (Q, P) maps of the encoder output are not image-sized."""
        if not getattr(explainer, "uses_tc", False):
            raise ValueError("AblationExperiments drives the tensor-core encoder: it needs a VGG-style encoder and "
                             "precision='fp32' or 'bf16'")
        self.ex = explainer
        self.num_delete_patches = int(num_delete_patches)
        self.patch_size = int(patch_size)
        self.num_delete_words = int(num_delete_words)
        self.chunk = int(chunk)

    # ------------------------------------------------------------------ evaluation.py:57-80
    def block_image(self, relevance):
        """relevance (H, W) -> mask (H, W), the reference's signature (one map)."""
        return ops.block_image(relevance.reshape(1, 1, *relevance.shape), self.num_delete_patches, self.patch_size)[0]

    def _teacher_forced_scores(self, feat, prefixes, words):
        """softmax score of ``words[i]`` as the next word after ``prefixes[i]`` (token lists starting with <start>) for
        the images with features ``feat`` (n,P,C): evaluation.py:139-142 (teacherforce_forward + softmax of the last row)."""
        dev = feat.device
        L = max(len(p) for p in prefixes)
        toks = torch.tensor([p + [0] * (L + 1 - len(p)) for p in prefixes], dtype=torch.long, device=dev)
        pred = self.ex.explainer_forward(feat, toks)["pred"]                          # (n, L, V)
        last = torch.tensor([len(p) - 1 for p in prefixes], device=dev)
        rows = pred[torch.arange(len(prefixes), device=dev), last]
        return torch.softmax(rows, dim=-1).gather(1, torch.as_tensor(words, device=dev).view(-1, 1))[:, 0]

    # ------------------------------------------------------------------ evaluation.py:120-150
    def image_ablation(self, imgs, tokens, heat, req_img, req_t, pred, beam_size=3, max_cap_length=20):
        """imgs (B,3,H,W), tokens (B,T+1) with column 0 = <start>, heat (Q,3,H,W) relevance of request q = (req_img[q],
        req_t[q]), pred (B,T,V) the explainer's logits.  -> dict: ``disappear`` (Q,) bool — the word is not in the new
        caption (:147-149); ``score_diff`` (Q,) original minus new softmax score, NaN where the word disappeared
        (:143-146); ``captions``: the Q new captions (token lists)."""
        ex = self.ex
        dev = ex.device
        eng = ex.engine()
        Q = heat.shape[0]
        req_img_l, req_t_l = req_img.tolist(), req_t.tolist()
        words = [int(tokens[b, t + 1]) for b, t in zip(req_img_l, req_t_l)]
        with torch.no_grad():
            _, masked = ops.block_image(heat, self.num_delete_patches, self.patch_size, images=imgs, req_img=req_img,
                                        want_mask=False)
            orig = torch.softmax(pred[req_img.long(), req_t.long()], dim=-1).gather(
                1, torch.tensor(words, device=dev).view(-1, 1))[:, 0]
            searcher = ex._searcher()
            caps, feats = [], []
            for q0 in range(0, Q, self.chunk):
                est = eng.forward(masked[q0:q0 + self.chunk])
                feat = eng.features(est, "pixel").clone()
                del est
                proj, glob = ex._search_inputs(feat)
                caps += searcher.search(proj, glob, ex.word_map, beam_size=beam_size, max_cap_length=max_cap_length)
                feats.append(feat)
            feat = torch.cat(feats)
            disappear = torch.tensor([w not in c for w, c in zip(words, caps)], device=dev)
            score_diff = torch.full((Q,), float("nan"), device=dev)
            keep = [q for q in range(Q) if words[q] in caps[q]]
            if keep:
                start = ex.word_map['<start>']
                prefixes = [[start] + caps[q][:caps[q].index(words[q])] for q in keep]
                idx = torch.tensor(keep, device=dev)
                new = self._teacher_forced_scores(feat[idx], prefixes, [words[q] for q in keep])
                score_diff[idx] = orig[idx] - new
        return dict(disappear=disappear, score_diff=score_diff, captions=caps, masked=masked)

    # ------------------------------------------------------------------ evaluation.py:344-447
    def bbox_correctness(self, heat, boxes, n_boxes=None, thresholds=(0, 0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9),
                         negative=False, inplace_quirk=True):
        """The pointing-game style score of ``bbox_experiment``: heat (Q,3,H,W), boxes (Q,nb,4) int (x0,y0,x1,y1) already
        scaled to the network's input size (:420-424) -> (Q, n_thr): per threshold the best share over the request's
        boxes of the positive relevance that lies inside a box (the reference keeps the maximum over the boxes of a
        category, :428-429).  ``inplace_quirk`` reproduces the reference's in-place thresholding (see ops.bbox_ratio)."""
        ratio = ops.bbox_ratio(heat, boxes, n_boxes=n_boxes, thresholds=thresholds, negative=negative,
                               inplace_quirk=inplace_quirk)
        return ratio.max(1).values

    # ------------------------------------------------------------------ evaluation.py:449-547
    @staticmethod
    def tpfp_statistics(heat, n_quantiles=100):
        """The per-word statistics ``tpfp_experiment`` records for true-/false-positive words (:503-513): of the channel
        mean of each heat-map (Q,3,H,W) -> dict of (Q,) tensors ``mean``, ``mean_abs``, ``mean_pos`` (sum of the positive
        part / number of positive pixels, 0 if none), ``max`` and ``quantile`` (Q, n_quantiles) at i/100 (numpy's default
        linear interpolation).  Device tensor ops (one sort per request); whether a word counts as TP or FP — membership
        in the reference captions' vocabulary, :469-470 — is the caller's bookkeeping."""
        m = heat.float().mean(1).flatten(1)                                        # np.mean(axis=(0,1)) -> (H*W)
        npos = (m > 0).sum(1)
        pos = m.clamp(min=0).sum(1)
        q = torch.arange(n_quantiles, device=m.device, dtype=m.dtype) / 100.0
        return dict(mean=m.mean(1), mean_abs=m.abs().mean(1),
                    mean_pos=torch.where(npos > 0, pos / npos.clamp(min=1), torch.zeros_like(pos)),
                    max=m.max(1).values, quantile=torch.quantile(m, q, dim=1).t().contiguous())

    @staticmethod
    def tpfp_split(tokens, frequent_ids, ref_encoded_caps, special_ids):
        """Which words of a predicted caption ``tpfp_experiment`` files under TP / FP (evaluation.py:462-481, :516):
        ``tokens`` = [<start>, w1, ..., wT]; a word counts if it is in ``frequent_ids`` (the reference's
        ``frequent_list``); it is a true positive if it occurs in any reference caption (``ref_encoded_caps``, lists of
        token ids; <start> / <pad> / <end> / <unk> = ``special_ids`` are dropped from that vocabulary), else a false
        positive.  -> (tp, fp): lists of word positions t (0-based, word t = tokens[t+1])."""
        special = set(int(v) for v in special_ids)
        vocab = {int(w) for cap in ref_encoded_caps for w in cap} - special
        frequent = set(int(v) for v in frequent_ids)
        tp = [t for t, w in enumerate(tokens[1:]) if int(w) in frequent and int(w) in vocab]
        fp = [t for t, w in enumerate(tokens[1:]) if int(w) in frequent and int(w) not in vocab]
        return tp, fp

    # ------------------------------------------------------------------ evaluation.py:234-262
    def word_ablation(self, feat, tokens, r_words, req_img, req_t, pred):
        """feat (B,P,C) encoder features, r_words (Q,T) linguistic relevance of each request (entry 0 = <start>).
        Deletes the ``num_delete_words`` most relevant preceding words (never <start>, :241-246) and returns the score
        drop of the explained word (Q,) under teacher forcing of the shortened prefix.  Requests need
        t >= num_delete_words (the reference uses t >= 6)."""
        dev = feat.device
        req_img_l, req_t_l = req_img.tolist(), req_t.tolist()
        if any(t < self.num_delete_words for t in req_t_l):
            raise ValueError("word ablation needs at least num_delete_words preceding words per request")
        toks = tokens.tolist()
        words = [toks[b][t + 1] for b, t in zip(req_img_l, req_t_l)]
        prefixes = []
        for q, (b, t) in enumerate(zip(req_img_l, req_t_l)):
            top = torch.topk(r_words[q, 1:t + 1], k=self.num_delete_words).indices.tolist()       # :241
            drop = {i + 1 for i in top}
            prefixes.append([w for i, w in enumerate(toks[b][:t + 1]) if i not in drop])          # np.delete (:246)
        with torch.no_grad():
            orig = torch.softmax(pred[req_img.long(), req_t.long()], dim=-1).gather(
                1, torch.tensor(words, device=dev).view(-1, 1))[:, 0]
            new = self._teacher_forced_scores(feat[req_img.long()], prefixes, words)
        return orig - new
