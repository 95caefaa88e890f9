"""GPU probe: caption a batch of images and explain every word of the captions, two ways, in one process.

  (a) ``model.beam_search_device(imgs)`` (the model's library encoder forward + the device search), then
      ``BatchExplainer.explain(imgs, tokens, words_per_image)`` (tensor-core encoder forward + explanation);
  (b) ``BatchExplainer.explain_images(imgs)``: one tensor-core encoder forward shared by the search and the explanation.

gridTD with VGG16 at 224x224, H = E = 512, V = 10 000, 64 images (bench.py's model and images), precision 'bf16' and
'mixed'.  A randomly initialised model never emits <end>, so both sides search with beam size 2 (the explainer's
get_hidden_parameters) and a fixed max_cap_length of 20: every caption has 19 words, 1216 requests per call.
The two run alternately after warm-up.  Per call: words explained per second (host clock around the whole call, search
included, ending in a device synchronise) and the CUDA-event time of the encoder forward(s), the search and the
explanation (events recorded around the library calls each side makes).  Prints the GPU name and power limit."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "lrp-imagecaptioning-pytorch_b200"), os.path.join(ROOT, "tests")):
    sys.path.insert(0, p)
import torch  # noqa: E402

import bench  # noqa: E402
from lrpx.pipeline import BatchExplainer  # noqa: E402


class Phases:
    """CUDA events around wrapped calls, summed per phase name."""

    def __init__(self):
        self.marks = []

    def wrap(self, obj, attr, phase):
        fn = getattr(obj, attr)

        def timed(*a, **k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*a, **k)
            e1.record()
            self.marks.append((phase, e0, e1))
            return out
        setattr(obj, attr, timed)

    def take(self):
        torch.cuda.synchronize()
        ms = {}
        for phase, e0, e1 in self.marks:
            ms[phase] = ms.get(phase, 0.0) + e0.elapsed_time(e1)
        self.marks = []
        return ms


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:               # the probe still runs; the line says what is missing
        q = f"{torch.cuda.get_device_name(0)}, power limit not read ({e!r})"
    return q


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--max-cap-length", type=int, default=20)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--precisions", default="bf16,mixed")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("caption_explain_probe needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    dev = torch.device("cuda")
    print(f"GPU: {gpu_info()}")
    results = {}
    for prec in a.precisions.split(","):
        args = argparse.Namespace(images=a.images, words=19, vocab=10000, precision=prec)
        model, ex, imgs, _ = bench.build_problem(args, dev, 0)
        imgs = imgs.to(dev)
        wm = ex.word_map
        k, L = ex.CAPTION_SEARCH[0], a.max_cap_length
        be = BatchExplainer(ex, chunk=128)
        ph = Phases()
        be.explain_images(imgs, max_cap_length=L)          # builds the engine and the explainer's searcher
        model.beam_search_device(imgs[:1], wm, beam_size=k, max_cap_length=L)     # builds the model's searcher
        eng = be.eng
        ph.wrap(model, "_encode", "encoder (library)")
        ph.wrap(eng, "forward", "encoder (tensor cores)")
        ph.wrap(eng, "features", "encoder (tensor cores)")
        ph.wrap(model._beam, "search", "search")
        ph.wrap(ex._searcher(), "search", "search")
        ph.wrap(ex, "_search_inputs", "search")
        ph.wrap(be, "_explain_encoded", "explanation")
        start = wm['<start>']

        def run_a():
            found = model.beam_search_device(imgs, wm, beam_size=k, max_cap_length=L)
            caps = [c[1] for c in found]
            T = max(len(c) for c in caps)
            toks = torch.tensor([[start] + c + [0] * (T - len(c)) for c in caps], dtype=torch.long, device=dev)
            heat, _ = be.explain(imgs, toks, words_per_image=[len(c) for c in caps])
            return caps, heat.shape[0]

        def run_b():
            res = be.explain_images(imgs, max_cap_length=L)
            return res.captions, res.heat.shape[0]

        runs = {"a": run_a, "b": run_b}
        for side in "abab":                                  # warm-up: every shape of the timed calls
            runs[side]()
        ph.take()
        rec = {"a": [], "b": []}
        caps = {}
        for _ in range(a.reps):
            for side in "ab":
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                caps[side], Q = runs[side]()
                torch.cuda.synchronize()
                wall = time.perf_counter() - t0
                rec[side].append(dict(wall_ms=wall * 1e3, words=Q, words_per_s=Q / wall, **ph.take()))
        med = lambda xs: sorted(xs)[len(xs) // 2]
        differ = sum(x != y for x, y in zip(caps["a"], caps["b"]))
        out = {}
        for side, label in (("a", "beam_search_device + explain"), ("b", "explain_images")):
            r = rec[side]
            keys = sorted({kk for x in r for kk in x})
            m = {kk: med([x.get(kk, 0.0) for x in r]) for kk in keys}
            out[side] = m
            phases = ", ".join(f"{kk} {m[kk]:.2f} ms" for kk in keys if kk not in ("wall_ms", "words", "words_per_s"))
            print(f"[{prec}] ({side}) {label}: {m['words']} words in {m['wall_ms']:.2f} ms = {m['words_per_s']:.0f} "
                  f"words/s (median of {a.reps}); {phases}")
        print(f"[{prec}] captions that differ between (a) and (b): {differ} of {a.images} images; "
              f"(b)/(a) words/s {out['b']['words_per_s'] / out['a']['words_per_s']:.3f}")
        results[prec] = dict(out, captions_differ=differ)
        del model, ex, be, eng
        torch.cuda.empty_cache()
    print(json.dumps(dict(gpu=gpu_info(), beam_size=2, max_cap_length=a.max_cap_length, images=a.images,
                          results=results)))


if __name__ == "__main__":
    main()
