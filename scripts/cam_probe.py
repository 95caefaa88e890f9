"""GPU probe: Grad-CAM and Guided Grad-CAM through lrpx.pipeline.BatchExplainer, next to the guided gradient.

Workload: bench.py's config-2 model and inputs — gridTD with VGG16 at 224x224, H = E = 512, V = 10 000, 64 images x 19
words = 1216 requests per call — in precision 'bf16' and 'fp32'.  Per precision, eager and graph-replayed:

  grad_cam                      ExplainGridTDGradCam: (Q, 196) maps, no encoder chain
  guided_grad_cam_full          ExplainGridTDGuidedGradCam, the CAM factor fused into the chain's last epilogue, fp32 (Q,3,H,W)
  guided_grad_cam_channel_mean  the same, delivered as the channel mean (Q,H,W)
  guided_gradient               ExplainiGridTDGuidedGradient: the chain-bound reference point
  unfused_guided_grad_cam       guided chain to fp32 (Q,3,H,W), then ops.cam_expand_mul over it in place: what the fusion
                                replaces (its maps are checked bit-equal to the fused ones)

and the per-image ``explain_caption`` loop of ExplainGridTDGradCam / ExplainGridTDGuidedGradCam on 2 images with their
19-word captions given (the caption search is not timed).  Prints explanations/s (CUDA events around ``--steps`` calls
after ``--warmup`` calls of the same shapes; the per-image loop: host clock ending in a device synchronise), the per-phase
CUDA-event ms of one eager call, and the GPU's name, power limit, maximum and current SM clock and power draw before and
after the runs."""
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
import synth  # noqa: E402
from lrpx import ops  # noqa: E402
from lrpx.pipeline import BatchExplainer  # noqa: E402


def gpu_state():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm,power.draw",
                               "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:               # the probe still runs; the line says what is missing
        return f"{torch.cuda.get_device_name(0)}, clock / power not read ({e!r})"


class Unfused(BatchExplainer):
    """Guided Grad-CAM without the fused factor: the guided chain writes the full fp32 gradient, then
    lrpx_cam_expand_mul_f32 reads it back and multiplies it (in place)."""

    def _explain_encoded(self, est, feat, tokens, req_img, req_t, heat, host=None):
        st = self.ex.explainer_forward(feat, tokens)
        req_word = tokens[req_img.long(), req_t.long() + 1].to(torch.int32)
        r_feat, r_words = self.ex._decode(st, req_img, req_t, req_word, self.tc_gemm, self.head_idx, self._dec_ws)
        fh, fw = est.feat_hw
        maps = ops.grad_cam(st["feat"], r_feat, req_img).view(-1, fh, fw)
        Kh, Kw = self.ex._expand_ops(fh, fw, int(est.x.shape[2]), int(est.x.shape[3]))
        self.eng.relevance(est, r_feat, req_img, chunk=self.chunk, out=heat)
        ops.cam_expand_mul(heat, maps, Kh, Kw, out=heat)
        return r_words, st["pred"], (maps, Kh, Kw)


class Phases:
    """CUDA events around wrapped calls of one eager call, summed per phase name (removed before graph capture)."""

    def __init__(self, hooks):
        self.hooks, self.saved, self.marks = hooks, [], []

    def __enter__(self):
        for obj, attr, phase in self.hooks:
            fn = getattr(obj, attr)
            self.saved.append((obj, attr, fn))

            def timed(*a, _fn=fn, _phase=phase, **k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                out = _fn(*a, **k)
                e1.record()
                self.marks.append((_phase, e0, e1))
                return out
            setattr(obj, attr, timed)
        return self

    def __exit__(self, *exc):
        for obj, attr, fn in reversed(self.saved):
            setattr(obj, attr, fn)
        self.saved = []

    def take(self):
        torch.cuda.synchronize()
        ms = {}
        for phase, e0, e1 in self.marks:
            ms[phase] = round(ms.get(phase, 0.0) + e0.elapsed_time(e1), 3)
        self.marks = []
        return ms


def timed_calls(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--images", type=int, default=64)
    ap.add_argument("--words", type=int, default=19)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--precisions", default="bf16,fp32")
    ap.add_argument("--per-image", type=int, default=2, help="images of the per-image explain_caption loop")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("cam_probe needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    from models import gridTDmodel as G
    dev = torch.device("cuda")
    state_before = gpu_state()
    print(f"GPU before: {state_before}", flush=True)
    V, H, E = 10000, 512, 512
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(1000, V, H, E), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(2000))
    model.to(dev).eval()
    ns = argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                            save_path=os.path.join("/tmp", "lrpx_cam_probe"), dataset="syn", weight="")
    imgs_h, toks_h = bench.problem_inputs(argparse.Namespace(images=a.images, words=a.words, vocab=V), 0)
    imgs, toks = imgs_h.to(dev), toks_h.to(dev)
    Q = a.images * a.words
    results = {}
    for prec in a.precisions.split(","):
        exs = {name: cls(ns, synth.word_map(V), model=model, precision=prec) for name, cls in
               (("cam", G.ExplainGridTDGradCam), ("ggc", G.ExplainGridTDGuidedGradCam),
                ("guided", G.ExplainiGridTDGuidedGradient))}
        methods = {"grad_cam": lambda g: BatchExplainer(exs["cam"], use_graph=g),
                   "guided_grad_cam_full": lambda g: BatchExplainer(exs["ggc"], use_graph=g),
                   "guided_grad_cam_channel_mean": lambda g: BatchExplainer(exs["ggc"], use_graph=g, deliver="channel_mean"),
                   "guided_gradient": lambda g: BatchExplainer(exs["guided"], use_graph=g),
                   "unfused_guided_grad_cam": lambda g: Unfused(exs["ggc"], use_graph=g)}
        res = {}
        outs = {}
        for name, make in methods.items():
            row = {}
            for graph in (False, True):
                be = make(graph)
                if not graph:                    # one eager call under the phase events (after a warm-up call)
                    be.explain(imgs, toks)
                    ex = be.ex
                    hooks = [(be.eng, "forward", "encoder forward"), (ex, "explainer_forward", "explainer forward"),
                             (ex, "_decode", "decoder gradient"), (ops, "grad_cam", "grad_cam"),
                             (ops, "cam_expand_rows", "cam_expand_rows"), (be.eng, "relevance", "encoder chain"),
                             (ops, "cam_expand_mul", "cam_expand_mul")]
                    with Phases(hooks) as ph:
                        be.explain(imgs, toks)
                        row["phase_ms"] = ph.take()
                heat = [None]

                def call():
                    heat[0] = be.explain(imgs, toks)[0]
                ms = timed_calls(call, a.steps, a.warmup)
                row["graph" if graph else "eager"] = dict(ms_per_call=round(ms, 3), explanations_per_s=round(Q / ms * 1e3, 1))
                if graph and name in ("guided_grad_cam_full", "unfused_guided_grad_cam"):
                    outs[name] = heat[0].clone()
                del be, heat
            res[name] = row
            print(f"[{prec}] {name}: eager {row['eager']['explanations_per_s']:.0f} /s ({row['eager']['ms_per_call']:.2f} ms), "
                  f"graph {row['graph']['explanations_per_s']:.0f} /s ({row['graph']['ms_per_call']:.2f} ms); "
                  f"phases (eager) {row['phase_ms']}", flush=True)
            torch.cuda.empty_cache()
        res["fused_equals_unfused"] = bool(torch.equal(outs["guided_grad_cam_full"], outs["unfused_guided_grad_cam"]))
        print(f"[{prec}] fused Guided Grad-CAM == unfused (bit for bit): {res['fused_equals_unfused']}", flush=True)
        del outs
        # the per-image API: explain_caption per image on its given 19-word caption
        for name in ("cam", "ggc"):
            ex = exs[name]
            n = min(a.per_image, a.images)

            def run_one(i):
                ex.preprocess_img = lambda path: imgs[i:i + 1]

                def given(path, beam_size, max_cap_length):
                    ex.beam_caption, ex.beam_caption_encode = ["(given)"], toks_h[i].tolist()
                    return None
                ex._find_caption = given
                ex.explain_caption(f"image{i}.jpg")
            run_one(0)                                   # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for i in range(n):
                run_one(i)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            key = "per_image_" + ("grad_cam" if name == "cam" else "guided_grad_cam")
            res[key] = dict(images=n, ms_per_image=round(wall / n * 1e3, 2), explanations_per_s=round(n * a.words / wall, 1))
            print(f"[{prec}] {key}: {res[key]}", flush=True)
        results[prec] = res
        del exs, methods
        torch.cuda.empty_cache()
    state_after = gpu_state()
    print(f"GPU after: {state_after}", flush=True)
    out = dict(gpu_before=state_before, gpu_after=state_after, images=a.images, words=a.words, requests=Q,
               steps=a.steps, warmup=a.warmup, results=results)
    print(json.dumps(out))
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
