#!/usr/bin/env python
"""bench.py — LRP explanations/s (image heat-map + linguistic relevance) on B200, with parity reported beside
every number.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--config C] [--precision P] [--deliver D]     one JSON line (rank 0)
  python bench.py --impl reference [--config C] ...        the reference itself on the host CPU cores: the UNMODIFIED
                                                           reference staged under baseline/_ref (oracle/stage_reference.py)
                                                           when present, else the oracle port

--config (BASELINE.json `configs`, 1-based; default 2 — the configuration the metric is quoted on):
  2  gridTD (VGG16 + adaptive-attention LSTM), 64 images x 19 caption words per GPU per step, alpha=1/beta=0 image +
     linguistic relevance of every word.  One step = encoder forward + per-layer gains (tcgen05) -> explainer
     teacher-forced forward -> decoder relevance for all requests -> encoder relevance chain (tcgen05) -> heat-maps.
  3  AoA decoder on 36 x 2048 bottom-up region features (AOAModelBU, H = E = 1024, 8 heads), beam size 3: device beam
     search + explainer forward + decoder relevance of every caption word (the explanation ends at the features).
  4  VGG16 encoder LRP only through LRPtools.compute_lrp: 512 (image, target relevance) requests per GPU per step.
  5  one lrp_tune training step (train.py:211-233) on gridTD, batch 128 per GPU, DDP gradient all-reduce over NCCL.
--precision: bf16 (tcgen05 chain with bf16 operands; the headline mode) | fp32 (the fp32-accurate mode: bf16x3 operands,
  fp32 gains, hi|lo storage — the reference's rtol 1e-4 bar on tensor cores) | mixed (fp32-accurate forward once per
  image, bf16 chain per explanation).
--method (config 2): lrp (default) | gradient | guided — the reference's comparison explainers (ExplainGridTDGradient /
  ExplainiGridTDGuidedGradient) through the same pipeline; device-resident timing + parity against the oracle's backward.
--deliver (config 2, end-to-end leg): full (Q,3,224,224 fp32, the reference's return value) | channel_mean
  ((Q,224,224): what evaluation.py:134,411,503 reduces every heat-map to) | fp16.

--dump-outputs DIR: after the timed steps, write what the timed call returned in its last step as DIR/<name>.npy
  (float32; float64 and integer arrays as float64), at most 64,000,000 bytes in all: an array too large for its share is
  written as a fixed, seeded sample of its elements plus the sampled flat positions (<name>_index.npy).  Inputs are seeded,
  so two builds run with the same arguments can be compared file by file.  Under torchrun: rank 0's shard.

Without --config the N = 1 run also measures configs 3, 4, 5, the mixed / fp32-accurate modes, the ResNet101 variant and
the gradient-family explainers of config 2 briefly and attaches them under "also" (each with its own parity figures), so that one driver run covers every configuration.
Under torchrun (N > 1) each rank works on its own shard (requests are independent: no collective on the data path;
config 5: DDP all-reduce); timing = CUDA events, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True          # bench.py writes nothing into the tree, not even __pycache__ of what it imports
ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "lrp-imagecaptioning-pytorch_b200")
for p in (PKG, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

METRIC = "lrp_explanations_per_s"
UNIT = "explanations/s"


def parse(argv=None):
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=0, choices=[0, 2, 3, 4, 5],
                    help="BASELINE.json configuration; 0 (default) = config 2 plus short 'also' runs of the others at N = 1")
    ap.add_argument("--precision", default=None, choices=["bf16", "fp32", "mixed"],
                    help="default: bf16 (config 5: fp32 — the fixed encoder's features at fp32 accuracy)")
    ap.add_argument("--deliver", default="full", choices=["full", "channel_mean", "fp16"])
    ap.add_argument("--encoder", default="vgg16", choices=["vgg16", "resnet101"],
                    help="config 2: the image encoder (resnet101: 7x7 grid of 2048-d features, bf16 chain of lrpx.tc_resnet)")
    ap.add_argument("--images", type=int, default=0, help="images (config 2/4: requests) per GPU per step; 0 = the config's size")
    ap.add_argument("--words", type=int, default=19, help="caption words per image (random-init captions run to max length)")
    ap.add_argument("--vocab", type=int, default=10000)
    ap.add_argument("--chunk", type=int, default=128, help="explanations per relevance-chain launch group")
    ap.add_argument("--no-graph", action="store_true", help="launch eagerly instead of replaying a CUDA graph of the step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-also", action="store_true")
    ap.add_argument("--library-encoder", action="store_true",
                    help="config 5: run the fixed VGG16 forward through the library convolutions instead of the tcgen05 engine")
    ap.add_argument("--method", default="lrp", choices=["lrp", "gradient", "guided"],
                    help="config 2: the explainer family (gradient / guided: the f4 explainers, device-resident timing only)")
    ap.add_argument("--profile-step", action="store_true",
                    help="run 1 warm-up + 1 step and exit (the command line captured under ncu for profiles/)")
    ap.add_argument("--cpu-words", type=int, default=19, help="words per image of the bounded CPU sample")
    ap.add_argument("--cpu-images", type=int, default=4, help="images of the bounded CPU sample (about 10-30 s of host work)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (at most 64 MB in all)")
    a = ap.parse_args(argv)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.also = (a.config == 0) and not a.no_also
    if a.config == 0:
        a.config = 2
    if a.images == 0:
        a.images = {2: 64, 3: 64, 4: 512, 5: 128}[a.config]
    if a.precision is None:
        a.precision = "fp32" if a.config == 5 else "bf16"
    return a


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        d = json.load(open(path))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, src="fallback")


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(index), "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, smax, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); smax = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


class Ctx:
    """rank / device / process-group plumbing + the timing contract (barrier + synchronize on both sides, CUDA
    events on the launching stream, max over ranks)."""

    def __init__(self):
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local = int(os.environ.get("LOCAL_RANK", 0))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: lrpx has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.numa = bind_to_gpu_numa_node(self.local)      # before any pinned allocation
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        torch.backends.cuda.matmul.allow_tf32 = False
        torch.backends.cudnn.allow_tf32 = False

    def barrier(self):
        if self.dist is not None:
            self.dist.barrier()
        torch.cuda.synchronize()

    def timed(self, fn, steps):
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        if self.dist is not None:
            t = torch.tensor([ms], device=self.dev)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def close(self):
        if self.dist is not None:
            self.dist.barrier()
            self.dist.destroy_process_group()

    def affinity(self):
        return f"{len(self.numa)} cores nearest to the GPU (NVML)" if isinstance(self.numa, list) else self.numa


def bind_to_gpu_numa_node(index):
    """Pins this rank's process to the CPU cores nearest to its GPU (NVML's ideal affinity) so that the pinned
    host buffers of the end-to-end path are first-touched on the GPU's own NUMA node."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        return sorted(os.sched_getaffinity(0))
    except Exception as e:      # affinity is an optimisation only
        return f"unavailable: {e!r}"


def write_outputs(dirname, arrays, budget=64_000_000, seed=0):
    """Writes each tensor of `arrays` (name -> tensor) as <dirname>/<name>.npy: float64 and integer tensors as float64
    (integers are exact below 2**53), the others as float32.  The files, .npy headers included, stay within `budget`
    bytes: every array gets an equal share; one larger than its share is written as the elements at a fixed, seeded set
    of flat positions, which go to <name>_index.npy (float64), so that the same arguments always select the same elements."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    share = budget // len(arrays) - 1024                # 1024: room for the headers of the array's two files
    for name, t in arrays.items():
        t = t.detach()
        t = t.double() if t.dtype == torch.float64 or not t.is_floating_point() else t.float()
        flat = t.reshape(-1)
        if flat.numel() * flat.element_size() > share:
            k = share // (flat.element_size() + 8)
            idx = torch.unique(torch.randint(0, flat.numel(), (k,), generator=torch.Generator().manual_seed(seed)))
            np.save(os.path.join(dirname, name + "_index.npy"), idx.double().numpy())
            t = flat[idx.to(flat.device)]
        np.save(os.path.join(dirname, name + ".npy"), t.cpu().numpy())


def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import lrp_oracle as O
    return O


def _ref_runner():
    """The staged reference (baseline/_ref or /root/reference), or None."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import ref_runner
        return ref_runner if ref_runner.available() else None
    except Exception:
        return None


def spearman(a, b):
    a, b = a.detach().double().flatten().cpu(), b.detach().double().flatten().cpu()
    ra = torch.empty_like(a); ra[a.argsort()] = torch.arange(a.numel(), dtype=torch.double)
    rb = torch.empty_like(b); rb[b.argsort()] = torch.arange(b.numel(), dtype=torch.double)
    ra -= ra.mean(); rb -= rb.mean()
    return float((ra * rb).sum() / (ra.norm() * rb.norm()))


# =================================================================================================== config 2
def build_problem(args, device, seed):
    """Random-init gridTD/VGG16 model + synthetic images and captions (seeded, SURVEY.md §8d)."""
    import argparse as ap
    import synth
    from models import gridTDmodel as G
    V, H, E = args.vocab, 512, 512
    torch.manual_seed(seed)
    enc = getattr(args, "encoder", "vgg16")
    if enc == "resnet101":
        model = G.GridTDModel(E, H, V, "resnet101", n_pixel=49)
        model.load_state_dict(synth.gridtd_decoder_state(1000 + seed, V, H, E, C=2048, n_pixel=49), strict=False)
        g = torch.Generator().manual_seed(2000 + seed)
        for m in model.img_encoder.encoder.modules():            # kaiming-normal convs (constructor) + non-trivial BatchNorm statistics
            if isinstance(m, torch.nn.BatchNorm2d):
                m.running_mean.copy_(torch.randn(m.num_features, generator=g) * 0.2)
                m.running_var.copy_(torch.rand(m.num_features, generator=g) + 0.5)
                m.weight.data.copy_(torch.rand(m.num_features, generator=g) + 0.5)
                m.bias.data.copy_(torch.randn(m.num_features, generator=g) * 0.2)
    else:
        model = G.GridTDModel(E, H, V, "vgg16")
        model.load_state_dict(synth.gridtd_decoder_state(1000 + seed, V, H, E), strict=False)
        model.img_encoder.encoder.load_state_dict(synth.vgg_state(2000 + seed))
    if device is not None:
        model.to(device)
    model.eval()
    ns = ap.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder=enc, height=224, width=224,
                      save_path="/tmp/lrpx_bench", dataset="syn", weight="")
    ex = G.ExplainGridTDAttention(ns, synth.word_map(V), model=model, precision=getattr(args, "precision", "bf16"))
    imgs, toks = problem_inputs(args, seed)
    return model, ex, imgs, toks


def problem_inputs(args, seed):
    B, T, V = args.images, args.words, args.vocab
    g = torch.Generator().manual_seed(3000 + seed)
    imgs = torch.randn(B, 3, 224, 224, generator=g)
    toks = torch.randint(1, V - 4, (B, T + 1), generator=g)
    toks[:, 0] = V - 2
    return imgs, toks


_REF_CACHE = {}


def cpu_config2(args, seed, nimg, nwords, keep=False, use_reference=True):
    """The reference's per-word formulation on the host cores for the first `nimg` images of rank `seed`'s batch, the
    last `nwords` words of each: the UNMODIFIED reference when it is staged (kind "reference"), else the oracle port.
    keep=True also returns the heat-maps / word relevances / feature relevances it produced (the parity checker)."""
    import synth
    O = _oracle()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    V, H, E = args.vocab, 512, 512
    p = synth.gridtd_decoder_state(1000 + seed, V, H, E)
    vsd = synth.vgg_state(2000 + seed)
    a2 = argparse.Namespace(**vars(args)); a2.images = max(args.images, nimg)
    imgs, toks = problem_inputs(a2, seed)
    T = args.words
    words = list(range(T - nwords, T))
    rr = _ref_runner() if use_reference else None
    out = {} if keep else None
    t0 = time.perf_counter()
    if rr is not None:
        key = (seed, V)
        if key not in _REF_CACHE:                 # model construction is not part of the timed work
            _REF_CACHE[key] = rr.GridTDReference(p, vsd, V, H, E, synth.word_map(V))
        ref = _REF_CACHE[key]
        t0 = time.perf_counter()
        for b in range(nimg):
            img = imgs[b:b + 1]
            ref.set_image(img, toks[b].tolist())
            for t in words:
                heat, rw, rf = ref.explain_word(img, t)
                if keep:
                    out[(b, t)] = (heat[0], rw, rf[0].reshape(512, -1).t())
        kind = "reference"
    else:
        layers = O.vgg_layers_from_state(vsd)
        for b in range(nimg):
            img = imgs[b:b + 1]
            feats = O.sequential_forward(layers, img)[-1]
            st = O.gridtd_explainer_forward(p, feats[0], toks[b].tolist())
            for t in words:
                rf, rw, _ = O.gridtd_explain_wordt(p, st, t)
                heat = O.sequential_lrp(layers, img, rf.t().reshape(1, 512, 14, 14))
                if keep:
                    out[(b, t)] = (heat[0], rw, rf)
        kind = "port"
    dt = time.perf_counter() - t0
    what = ("the UNMODIFIED reference (ExplainGridTDAttention.explain_caption_wordt + explain_cnn, staged copy)"
            if kind == "reference" else "oracle port of the reference's per-word formulation")
    res = {"value": nimg * len(words) / dt, "unit": UNIT, "cores": cores, "kind": kind,
           "sample": f"{nimg} images (explainer forward once each) x {len(words)} words (decoder + VGG16 encoder "
                     f"relevance), {what}, fp32 torch-CPU, {dt:.2f} s"}
    return (res, out) if keep else res


def parity_config2(args, ex, eng, W, imgs_d, toks_d, heat, r_words, ref_out, T):
    """Parity of the timed run's OUTPUT against what the CPU leg computed for the same requests (same seeds):
    heat-maps (Spearman / rel-L2 / scale-relative max error), word relevances, and — decoder isolated — the decoder
    kernels against the oracle on the product's own encoder features; predicted-word arg-max; per-layer conservation."""
    from lrpx import ops
    import helpers
    O = _oracle()
    import synth
    sp, l2, mx, wd = [], [], [], []
    for (b, t), (h_ref, rw_ref, _) in ref_out.items():
        q = b * T + t
        a, r = heat[q].detach().cpu().double(), h_ref.double()
        sp.append(spearman(a, r))
        l2.append(float((a - r).norm() / r.norm()))
        mx.append(float((a - r).abs().max() / r.abs().max()))
        wd.append(float((r_words[q, :t + 1].detach().cpu().double() - rw_ref.double()).abs().max()))
    med = lambda v: sorted(v)[len(v) // 2]
    out = {"requests_checked": len(ref_out), "against": "reference" if _ref_runner() is not None else "oracle port",
           "heatmap_spearman_min": min(sp), "heatmap_spearman_median": med(sp),
           "heatmap_rel_l2_max": max(l2), "heatmap_rel_l2_median": med(l2),
           "heatmap_max_err_over_max_abs": max(mx), "words_max_abs": max(wd), "words_max_abs_median": med(wd),
           "note": "end to end against the fp32 reference: encoder features -> decoder (LSTM chain over the caption) -> "
                   "decoder relevance -> encoder chain; `decoder_*` isolate the decoder kernels on identical features"}
    # ---- decoder isolated: product decoder kernels vs the oracle decoder on the SAME (product) encoder features
    seed = 0
    p = synth.gridtd_decoder_state(1000 + seed, args.vocab, 512, 512)
    est = eng.forward(imgs_d[:1], keep_act=True)
    feat = eng.features(est, "pixel")
    st = ex.explainer_forward(feat, toks_d[:1])
    ts = torch.arange(T, dtype=torch.int32, device=feat.device)
    r_feat, rw = ops.gridtd_decoder_lrp(st, W, torch.zeros_like(ts), ts, toks_d[0, 1:].to(torch.int32), tc_gemm=True)
    fmap = feat[0].t().reshape(512, 14, 14).cpu()
    ost = O.gridtd_explainer_forward(p, fmap, toks_d[0].tolist())
    dmax, wmax = 0.0, 0.0
    for t in (0, T // 2, T - 1):
        rf, rwo, _ = O.gridtd_explain_wordt(p, ost, t)
        dmax = max(dmax, float((r_feat[t].cpu().double() - rf.double()).abs().max() / rf.double().abs().max()))
        wmax = max(wmax, float((rw[t, :t + 1].cpu().double() - rwo.double()).abs().max()))
    out["decoder_scale_rel_max"] = dmax
    out["decoder_words_max_abs"] = wmax
    out["argmax_bit_exact"] = bool(torch.equal(st["pred"][0].argmax(-1).cpu(), ost["pred"].argmax(-1)))
    # ---- conservation per layer (sum R at the input of every conv / sum R handed to the encoder output)
    trace = eng.conservation(est, r_feat, torch.zeros(T, dtype=torch.int32, device=feat.device))
    top = trace[0][1]
    out["conservation_per_layer"] = [round(v / top, 6) for _, v in trace[1:]]
    out["conservation_note"] = ("sum R_in / sum R at the encoder output for the 13 conv layers, top to bottom, over "
                                f"the {T} requests of image 0 (alpha=1/beta=0 without bias conserves up to the relevance "
                                "dropped where z+ == 0 or a pooled maximum is 0)")
    return out


def parity_resnet(args, model, ex, eng, W, imgs_d, toks_d, T):
    """ResNet101 variant of config 2: the encoder chain of the timed path against the oracle's restatement of the
    reference's ResNet rules (lrp_modules.py:197-280, fp64 on the host) for two requests of image 0, with the
    product decoder's own feature relevance as the target (the decoder kernels are pinned by the VGG variant)."""
    from lrpx import ops
    O = _oracle()
    est = eng.forward(imgs_d[:1])
    feat = eng.features(est, "pixel")
    st = ex.explainer_forward(feat, toks_d[:1])
    ts = torch.tensor([0, T - 1], dtype=torch.int32, device=feat.device)
    r_feat, _ = ops.gridtd_decoder_lrp(st, W, torch.zeros_like(ts), ts, toks_d[0, 1:][ts.long()].to(torch.int32),
                                       tc_gemm=True)
    heat = eng.relevance(est, r_feat, torch.zeros_like(ts))
    sd = {k: (v.detach().cpu().double() if v.is_floating_point() else v.detach().cpu())
          for k, v in model.img_encoder.encoder.state_dict().items()}
    fh, fw = est.feat_hw
    t0 = time.perf_counter()
    tgt = r_feat.cpu().double().transpose(1, 2).reshape(2, -1, fh, fw)
    ref = O.resnet_lrp(sd, imgs_d[:1].cpu().double().expand(2, -1, -1, -1), tgt)
    dt = time.perf_counter() - t0
    a = heat.cpu().double()
    par = {"requests_checked": 2, "against": "oracle port (fp64) of the ResNet rules, same feature relevance in",
           "heatmap_spearman_min": min(spearman(a[i], ref[i]) for i in range(2)),
           "heatmap_rel_l2_max": max(float((a[i] - ref[i]).norm() / ref[i].norm()) for i in range(2)),
           "conservation_sum_rin_over_sum_rout": [float(a[i].sum() / tgt[i].sum()) for i in range(2)]}
    cb = {"value": 2 / dt, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
          "sample": f"2 requests, ResNet101 encoder relevance only (oracle port, fp64 torch-CPU), {dt:.2f} s"}
    return cb, par


def run_config2(args, ctx, brief=False):
    from lrpx import ops, _lib
    from lrpx.pipeline import BatchExplainer
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    model, ex, imgs_h, toks_h = build_problem(args, dev, seed=rank)
    B, T = args.images, args.words
    Q = B * T
    eng = ex.engine()
    W = ex._lrp_weights()
    imgs_h = imgs_h.pin_memory()
    toks_h = toks_h.pin_memory()
    req_img = torch.arange(B, dtype=torch.int32).repeat_interleave(T).to(dev)
    req_t = torch.arange(T, dtype=torch.int32).repeat(B).to(dev)
    heat = torch.empty(Q, 3, 224, 224, device=dev, dtype=torch.float32)          # device-resident leg: the full fp32 maps
    deliver = args.deliver
    if deliver == "channel_mean":
        heat_h = torch.empty(Q, 224, 224, dtype=torch.float32).pin_memory()
    elif deliver == "fp16":
        heat_h = torch.empty(Q, 3, 224, 224, dtype=torch.float16).pin_memory()
    else:
        heat_h = torch.empty(Q, 3, 224, 224, dtype=torch.float32).pin_memory()
    heat_dv = heat if deliver == "full" else torch.empty(tuple(heat_h.shape), device=dev, dtype=heat_h.dtype)
    words_h = torch.empty(Q, T, dtype=torch.float32).pin_memory()
    imgs_d, toks_d = imgs_h.to(dev), toks_h.to(dev)
    ev = lambda: torch.cuda.Event(enable_timing=True)
    tc_gemm = True                    # decoder GEMMs as bf16x3 on tensor cores in both chain modes (BatchExplainer's default)
    pipe = BatchExplainer(ex, chunk=args.chunk, use_graph=not args.no_graph, tc_gemm=tc_gemm)
    pipe_e2e = pipe if deliver == "full" else BatchExplainer(ex, chunk=args.chunk, use_graph=not args.no_graph,
                                                             tc_gemm=tc_gemm, deliver=deliver)
    last = {}

    def step(imgs, toks):
        """The public batched call (lrpx.pipeline.BatchExplainer.explain)."""
        last["out"] = pipe.explain(imgs, toks, out=heat)

    def step_e2e():
        """Same call with HOST buffers: pinned images/captions in, pinned heat-maps / word relevances out."""
        pipe_e2e.explain(imgs_h, toks_h, out=heat_dv, host_out=(heat_h, words_h))

    if args.profile_step:
        step(imgs_d, toks_d)
        torch.cuda.synchronize()
        step(imgs_d, toks_d)
        torch.cuda.synchronize()
        print(json.dumps({"profile_step": "done", "explanations": Q}))
        return None

    def breakdown():
        """One instrumented step (outside the timed region): CUDA-event time of each phase."""
        marks = [ev() for _ in range(6)]
        calls0 = dict(_lib.CALLS)
        marks[0].record()
        est = eng.forward(imgs_d); marks[1].record()
        feat = eng.features(est, "pixel")
        st = ex.explainer_forward(feat, toks_d); marks[2].record()
        r_feat, r_words = ops.gridtd_decoder_lrp(st, W, req_img, req_t, toks_d[:, 1:].reshape(-1).to(torch.int32),
                                                 tc_gemm=tc_gemm)
        marks[3].record()
        eng.relevance(est, r_feat, req_img, chunk=args.chunk, out=heat); marks[4].record()
        torch.cuda.synchronize()
        names = ["encoder_forward_gains", "explainer_forward", "decoder_relevance", "encoder_relevance_chain"]
        calls = {k: _lib.CALLS[k] - calls0.get(k, 0) for k in _lib.CALLS}
        return {n: round(marks[i].elapsed_time(marks[i + 1]), 3) for i, n in enumerate(names)}, calls

    # eager warm-up + the instrumented step BEFORE any graph exists (a captured graph pins a private memory pool,
    # which would distort eager timings taken after it)
    eager = BatchExplainer(ex, chunk=args.chunk, use_graph=False, tc_gemm=tc_gemm)
    for _ in range(2):
        eager.explain(imgs_d, toks_d, out=heat)
    phase_ms, calls = breakdown()
    for _ in range(1 if brief else 2):                       # per-phase minimum of the instrumented steps
        again, _ = breakdown()
        phase_ms = {k: min(v, again[k]) for k, v in phase_ms.items()}
    del eager
    steps = args.steps
    for _ in range(max(args.warmup, 3)):
        step(imgs_d, toks_d)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    ms = ctx.timed(lambda: step(imgs_d, toks_d), steps)
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:          # before the end-to-end leg overwrites `heat`
        write_outputs(args.dump_outputs, {"heatmaps": last["out"][0], "word_relevance": last["out"][1]})
    # the chain's share of the TIMED (graph-replayed) step: chain_ms_in_step = ms_per_step - (the other phases)
    others = phase_ms["encoder_forward_gains"] + phase_ms["explainer_forward"] + phase_ms["decoder_relevance"]
    chain_in_step = max(ms / steps - others, phase_ms["encoder_relevance_chain"])
    r_words_last = last["out"][1]
    heat_last = heat.clone() if rank == 0 and not args.no_cpu_baseline and world == 1 else None
    for _ in range(2):
        step_e2e()
    ms_e2e = ctx.timed(step_e2e, steps)
    step_eager_ms = sum(phase_ms.values())
    # the same end-to-end call delivering channel-mean maps (what evaluation.py consumes): 3x fewer bytes to the host
    e2e_cm = None
    if deliver == "full" and not brief:
        cm_h = torch.empty(Q, 224, 224, dtype=torch.float32).pin_memory()
        cm_d = torch.empty(Q, 224, 224, device=dev, dtype=torch.float32)
        pipe_cm = BatchExplainer(ex, chunk=args.chunk, use_graph=not args.no_graph, tc_gemm=tc_gemm, deliver="channel_mean")
        step_cm = lambda: pipe_cm.explain(imgs_h, toks_h, out=cm_d, host_out=(cm_h, words_h))
        for _ in range(2):
            step_cm()
        ms_cm = ctx.timed(step_cm, steps)
        e2e_cm = {"value": world * Q * steps / (ms_cm * 1e-3), "unit": UNIT, "ms_per_step": ms_cm / steps,
                  "h2d_bytes_per_step": imgs_h.numel() * 4 + toks_h.numel() * 8,
                  "d2h_bytes_per_step": cm_h.numel() * 4 + words_h.numel() * 4, "deliver": "channel_mean"}
        del pipe_cm

    # launches of OUR kernels inside the timed region: one per C-ABI call, except the decoder call which
    # enqueues init + per step (3 element-wise kernels that also write the split GEMM operand + 2 tensor-core GEMMs)
    # + 8 tail kernels (csrc/decoder.cu; the 4 weight conversions run once, in the warm-up call that fills the persistent
    # workspace — LRPX_DEC_W3_READY afterwards)
    launches = sum(v for k, v in calls.items() if k != "lrpx_gridtd_decoder_lrp_f32")
    launches += calls.get("lrpx_gridtd_decoder_lrp_f32", 0) * (1 + 5 * T + 8)
    launches *= steps

    out = None
    if rank == 0:
        pk = peaks()
        total = world * Q * steps
        flops_alg = eng.flops_per_explanation()
        flops_mma = eng.mma_flops_per_explanation()
        ach_eager = flops_mma * Q / (phase_ms["encoder_relevance_chain"] * 1e-3) / 1e12
        ach_step = flops_mma * Q / (chain_in_step * 1e-3) / 1e12
        d2h = heat_h.numel() * heat_h.element_size() + words_h.numel() * 4
        out = {
            "metric": METRIC, "value": total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": {"bf16": "bf16", "mixed": "bf16 chain on a bf16x3 (fp32-accurate) forward"}.get(
                ex.precision, "bf16x3 (fp32-accurate)"),
            "data": "synthetic",
            "config": {"workload": "config 2: gridTD VGG16 LRP alpha1beta0 image+linguistic explanations, "
                                   f"{B} images x {T} words per GPU per step, 224x224, V={args.vocab}, H=E=512",
                       "baseline_config": 2, "precision": ex.precision, "deliver": deliver,
                       "explanations_per_step_per_gpu": Q, "chunk": args.chunk,
                       "host_affinity": ctx.affinity(), "cuda_graph": not args.no_graph,
                       "parallelism": f"request-sharded x{world}",
                       "l2": "working set (gains 1.9 GB + chain buffers) far larger than the 126 MB L2; no flush needed",
                       "decoder_relevance_dtype": ("f32 element-wise, GEMMs as error-compensated bf16x3 on tensor cores (f32 accumulate)"
                                                   if tc_gemm else "f32 (CUDA-core GEMMs)"),
                       "encoder_relevance_dtype": ("bf16 operands, f32 accumulate" if ex.precision in ("bf16", "mixed") else
                                                   "bf16x3 error-compensated operands (hi|lo storage, fp32 gains), f32 accumulate")},
            "e2e": {"value": total / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / steps,
                    "h2d_bytes_per_step": imgs_h.numel() * 4 + toks_h.numel() * 8,
                    "d2h_bytes_per_step": d2h, "deliver": deliver},
            "e2e_channel_mean": e2e_cm,
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": {"bound": "tensor", "kernel": "tc_conv_slab_kernel (encoder relevance chain)",
                         "achieved": ach_step, "peak": pk["tf_sustained"], "unit": "TFLOP/s",
                         "frac": ach_step / pk["tf_sustained"],
                         "achieved_note": "tensor-core FLOPs the chain executes per step / the chain's time INSIDE the timed "
                                          "graph-replayed step (ms_per_step minus the CUDA-event times of the other three "
                                          "phases); `achieved_eager` is the same over the chain's own CUDA-event time in an "
                                          "instrumented eager step",
                         "achieved_eager": ach_eager, "frac_eager": ach_eager / pk["tf_sustained"],
                         "traffic": chain_traffic(args.chunk) if ex.precision in ("bf16", "mixed") else None,
                         "traffic_note": "dram read+write bytes of the 13 chain layers per chunk of explanations (ncu --set "
                                         "full, profiles/r2_chain_full.md); algorithmic FLOPs per chunk = chunk x "
                                         "algorithmic_gflop_per_explanation",
                         "peak_source": pk["src"] + " sustained bf16",
                         "share_of_step": chain_in_step / (ms / steps),
                         "algorithmic_gflop_per_explanation": flops_alg / 1e9,
                         "executed_gflop_per_explanation": flops_mma / 1e9,
                         "reference_formulation_gflop_per_explanation": 2.0 * flops_alg / 1e9},
        }
        out["breakdown_ms"] = phase_ms
        is_resnet = getattr(args, "encoder", "vgg16") == "resnet101"
        if is_resnet:
            out["config"]["workload"] = out["config"]["workload"].replace("gridTD VGG16", "gridTD ResNet101 (7x7 x 2048 features)")
            out["roofline"]["kernel"] = "tc_conv_kernel / tc_conv_slab_kernel <MULX> (ResNet101 relevance chain, ~100 GEMMs)"
        if not brief and not is_resnet:
            try:
                out["roofline"]["layers"] = layer_table(eng, args.chunk, dev, pk, requests=Q)
            except Exception as e:  # never lose the bench line to the per-layer microbenchmark
                out["roofline"]["layers_error"] = repr(e)
        if not args.no_cpu_baseline and world == 1 and is_resnet:
            try:
                out["cpu_baseline"], out["parity"] = parity_resnet(args, model, ex, eng, W, imgs_d, toks_d, T)
            except Exception as e:
                out["parity"] = {"error": repr(e)}
        elif not args.no_cpu_baseline and world == 1:
            nimg = 1 if brief else max(1, args.cpu_images)
            nwords = max(1, min(args.cpu_words, T)) if not brief else min(4, T)
            cb, ref_out = cpu_config2(args, 0, nimg, nwords, keep=True)
            out["cpu_baseline"] = cb
            try:
                out["parity"] = parity_config2(args, ex, eng, W, imgs_d, toks_d, heat_last, r_words_last, ref_out, T)
            except Exception as e:
                out["parity"] = {"error": repr(e)}
    return out


def chain_traffic(chunk):
    """dram__bytes_read.sum + dram__bytes_write.sum of the relevance-chain launches, per `chunk` explanations, from the
    committed ncu --set full capture of all chain launches of one step; None if absent."""
    for name in ("r2_chain_full.json", "r1_chain_full.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            d = json.load(open(path))
            if d.get("dram_bytes_per_explanation"):
                return d["dram_bytes_per_explanation"] * chunk
    return None


def layer_table(eng, chunk, dev, pk, requests=None):
    """Per-layer achieved TFLOP/s of the relevance-chain launches (CUDA events, 5 launches each) at the launch sizes the
    engine uses: the low-resolution layers over all `requests` of a step in one launch (TcVggEngine.relevance_head),
    the others per chunk; `ms` is per chunk of explanations either way.  FLOPs = the tensor-core FLOPs executed."""
    from lrpx import tc
    rows = []
    x = torch.randn(1, 3, eng.convs[0].h, eng.convs[0].w, device=dev)
    st = eng.forward(x[:1])
    L = len(eng.convs)
    Q = requests or chunk
    n_wide = 0                                  # the engine's own rule (relevance_head): 2 GB per stage-1 buffer
    if Q > chunk:
        for li in range(L - 1, 0, -1):
            c, below = eng.convs[li], eng.convs[li - 1]
            oh, ow = (2 * c.h, 2 * c.w) if below.pool_after else (c.h, c.w)
            if max(tc.pf_rows(Q, c.h, c.w) * c.cout, tc.pf_rows(Q, oh, ow) * c.cin) * 2 * eng.rm > (2 << 30):
                break
            n_wide += 1
    for li in range(L - 1, -1, -1):
        c = eng.convs[li]
        n = Q if li >= L - n_wide else chunk
        rimg = torch.zeros(n, dtype=torch.int32, device=dev)
        a = torch.randn(tc.pf_rows(n, c.h, c.w), c.cout * eng.rm, device=dev).to(torch.bfloat16)
        bufs = [None, None]
        if li == 0:
            out = torch.empty(n, 3, c.h, c.w, device=dev)
            if eng.general:
                fn = lambda: tc.tc_conv(a, c.w_rel3, n, c.h, c.w, c.cout * eng.km, 24, 3, tc.EPI_INPUT3, out, row_img=rimg,
                                        x=st.x, a_phys=c.cout * eng.rm if eng.split else 0)
            elif c.w_rel3 is not None:          # the engine's own choice: filter columns folded into N
                fn = lambda: tc.tc_conv(a, c.w_rel3, n, c.h, c.w, c.cout, 24, 3, tc.EPI_INPUT3, out, row_img=rimg, x=st.x)
            else:
                fn = lambda: tc.tc_conv(a, c.w_rel, n, c.h, c.w, c.cout, 16, 3, tc.EPI_INPUT, out, row_img=rimg, x=st.x)
        else:
            below = eng.convs[li - 1]
            oh, ow = (2 * c.h, 2 * c.w) if below.pool_after else (c.h, c.w)
            bufs[1] = torch.empty(tc.pf_rows(n, oh, ow) * c.cin * eng.rm, device=dev, dtype=torch.bfloat16)
            fn = lambda: eng._run_layers(st, a, n, rimg, li, li + 1, bufs, 0)
        flops = 2.0 * n * c.h * c.w * c.cin * c.cout * 9 * eng.km
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 5
        rows.append({"layer": li, "hw": c.h, "k": 9 * c.cout * eng.km, "n": c.cin if li else 6, "launch_requests": n,
                     "ms": round(ms * chunk / n, 4), "tflops": round(flops / (ms * 1e-3) / 1e12, 1)})
        del a, bufs
    return rows


# =================================================================================================== config 3
def build_config3(args, dev, seed):
    import synth
    from models import aoamodel as A
    V, H, E = args.vocab, 1024, 1024
    model = A.AOAModelBU(E, H, 8, V, "bu")
    model.load_state_dict(synth.aoa_bu_state(97 + seed, V, H, E), strict=True)
    ns = argparse.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="bu", height=224, width=224,
                            save_path="/tmp/lrpx_bench", dataset="syn", weight="")
    ex = A.ExplainAOAAttention(ns, synth.word_map(V), model=model.to(dev).eval(), precision=args.precision)
    feats = synth.bu_features(98 + seed, args.images)
    return model, ex, feats


def run_config3(args, ctx, brief=False):
    """AoA decoder on bottom-up features, beam 3 (aoamodel.py:1064-1163 batched): explain_region_features_batch."""
    import synth
    from lrpx import _lib
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    model, ex, feats_h = build_config3(args, dev, seed=rank)
    feats_h = feats_h.pin_memory()
    feats_d = feats_h.to(dev)
    head = 3
    r = ex.explain_region_features_batch(feats_d, head)
    Q = int(r[0].shape[0])
    rf_h = torch.empty(tuple(r[0].shape), dtype=torch.float32).pin_memory()
    rw_h = torch.empty(tuple(r[1].shape), dtype=torch.float32).pin_memory()
    last = {}

    def step():
        last["r"] = ex.explain_region_features_batch(feats_d, head)

    def step_e2e():
        rr = ex.explain_region_features_batch(feats_h.to(dev, non_blocking=True), head)
        rf_h.copy_(rr[0], non_blocking=True)
        rw_h.copy_(rr[1], non_blocking=True)

    steps = args.steps
    for _ in range(max(args.warmup, 3)):
        step()
    calls0 = dict(_lib.CALLS)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    ms = ctx.timed(step, steps)
    clocks = sampler.stop() if sampler else None
    calls = {k: _lib.CALLS[k] - calls0.get(k, 0) for k in _lib.CALLS}
    if args.dump_outputs and rank == 0:
        r_feat, r_words, req_img, req_t, caps = last["r"]
        cap_len = max(len(c) for c in caps)
        captions = torch.tensor([[int(w) for w in c] + [-1] * (cap_len - len(c)) for c in caps])  # -1: past the end
        write_outputs(args.dump_outputs, {"feature_relevance": r_feat, "word_relevance": r_words,
                                          "request_image": req_img, "request_word": req_t, "captions": captions})
    for _ in range(2):
        step_e2e()
    ms_e2e = ctx.timed(step_e2e, steps)
    # the decoder-relevance call alone (captions given), CUDA events: the part of the step that is this path's own
    caps = last["r"][4]
    T = max(len(c) for c in caps)
    toks = torch.tensor([[ex.word_map['<start>']] + c + [0] * (T - len(c)) for c in caps])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fn = lambda: ex.explain_region_features_batch(feats_d, head, tokens=toks)
    fn(); torch.cuda.synchronize()
    e0.record()
    for _ in range(5):
        fn()
    e1.record(); torch.cuda.synchronize()
    ms_given = e0.elapsed_time(e1) / 5
    out = None
    if rank == 0:
        pk = peaks()
        B, P, C = feats_h.shape
        H = 1024
        # algorithmic bytes of forward + relevance with the captions given: features read once, saved state of
        # the T steps written + read once, r_feat (Q,P,C) written once, weights read once
        state_bytes = 4 * B * T * (12 * H + 8 * P + args.vocab)
        alg_bytes = 4 * (B * P * C + Q * P * C + Q * T) + 2 * state_bytes
        ach = alg_bytes / (ms_given * 1e-3) / 1e9
        total = world * Q * steps
        out = {"metric": METRIC, "value": total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f32 element-wise; GEMMs bf16x3 (f32 accumulate)" if args.precision == "bf16" else "f32",
               "data": "synthetic",
               "config": {"workload": f"config 3: AOAModelBU on {B} sets of 36 x 2048 bottom-up region features per GPU per "
                                      f"step, H=E=1024, 8 heads, V={args.vocab}, device beam search (beam 3) + explainer "
                                      f"forward + decoder relevance of every caption word (head {head})",
                          "baseline_config": 3, "explanations_per_step_per_gpu": Q, "caption_words": T,
                          "precision": args.precision, "parallelism": f"request-sharded x{world}",
                          "l2": "inputs re-read from HBM each step: saved state + outputs (0.4 GB) exceed the 126 MB L2"},
               "e2e": {"value": total / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / steps,
                       "h2d_bytes_per_step": feats_h.numel() * 4,
                       "d2h_bytes_per_step": rf_h.numel() * 4 + rw_h.numel() * 4},
               "gpu_launches": sum(calls.values()),
               "gpu_launches_note": "C-ABI calls per timed region (each decoder-relevance call enqueues ~5 kernels per LSTM step)",
               "clocks": clocks,
               "roofline": {"bound": "hbm", "kernel": "explainer forward + lrpx_aoa_decoder_lrp_f32 (captions given)",
                            "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"],
                            "traffic": None, "ms": ms_given,
                            "note": "launch-latency bound: ~25 small kernels per LSTM step over 64 feature sets; the beam "
                                    "search (vocabulary GEMM per step, library) is the rest of the step"},
               "breakdown_ms": {"search_forward_relevance": ms / steps, "forward_relevance_captions_given": ms_given}}
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"], out["parity"] = cpu_config3(args, ex, feats_h, caps, last["r"], head, 1 if brief else 2)
    return out


def cpu_config3(args, ex, feats, caps, res, head, nimg):
    """Oracle port of ExplainAOAAttention.explain_caption_wordt on the region features (the reference has no
    Explain*BU class, SURVEY §8c(ii): the oracle is pinned by fixture aoa_dec_bu) for `nimg` feature sets, all words,
    with the captions the device beam search found; parity of the timed run's outputs against it."""
    import synth
    O = _oracle()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    V, H, E = args.vocab, 1024, 1024
    p = synth.aoa_bu_state(97, V, H, E)
    r_feat, r_words, req_img, req_t = res[0], res[1], res[2].cpu(), res[3].cpu()
    t0 = time.perf_counter()
    n, dmax, wmax = 0, 0.0, 0.0
    start = ex.word_map['<start>']
    for b in range(nimg):
        toks = [start] + list(caps[b])
        st = O.aoa_explainer_forward(p, feats[b].t().reshape(2048, 6, 6), toks, 8)
        for t in range(len(caps[b])):
            rf, rw, _ = O.aoa_explain_wordt(p, st, t, head)
            q = int(((req_img == b) & (req_t == t)).nonzero()[0])
            dmax = max(dmax, float((r_feat[q].cpu().double() - rf.double()).abs().max() / rf.double().abs().max()))
            wmax = max(wmax, float((r_words[q, :t + 1].cpu().double() - rw.double()).abs().max()))
            n += 1
    dt = time.perf_counter() - t0
    cb = {"value": n / dt, "unit": UNIT, "cores": cores, "kind": "port",
          "sample": f"{nimg} feature sets x all caption words ({n} explanations; explainer forward + decoder relevance, "
                    f"captions given), oracle port, fp32 torch-CPU, {dt:.2f} s"}
    par = {"requests_checked": n, "against": "oracle port (pinned by fixture aoa_dec_bu)",
           "decoder_scale_rel_max": dmax, "words_max_abs": wmax,
           "beam_indices": "bit-exact vs the reference's beam_search in tests/test_gpu_beam.py (fixture tune_bu)"}
    return cb, par


# =================================================================================================== config 4
def run_config4(args, ctx, brief=False):
    """VGG16 encoder LRP only, through the drop-in API: encoder.compute_lrp(images, target=R) (lrp_wrapper.py:63-87)
    on `images` requests per GPU per step — forward + gains once per request image, one contraction per layer."""
    import synth
    from models import vgg
    from LRPtools import lrp_wrapper
    from lrpx import _lib
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    n = args.images
    net = vgg.vgg16().features[0:-1]
    net.load_state_dict(synth.vgg_state(2000 + rank))
    net = net.to(dev).eval()
    lrp_wrapper.add_lrp(net)
    g = torch.Generator().manual_seed(4000 + rank)
    x_h = torch.randn(n, 3, 224, 224, generator=g).pin_memory()
    tgt_h = (torch.randn(n, 512, 14, 14, generator=g) * 1e-3).pin_memory()
    x_d, tgt_d = x_h.to(dev), tgt_h.to(dev)
    out_h = torch.empty(n, 3, 224, 224).pin_memory()
    os.environ["LRPX_NO_GRAD_ACCUMULATION"] = "1"       # throughput: a fresh sample per call (Q1 off on both arms)
    last = {}

    def step():
        last["rel"] = lrp_wrapper.compute_lrp(net, x_d, target=tgt_d, precision=args.precision)

    def step_e2e():
        rel = lrp_wrapper.compute_lrp(net, x_h.to(dev, non_blocking=True), target=tgt_h.to(dev, non_blocking=True),
                                      precision=args.precision)
        out_h.copy_(rel, non_blocking=True)

    steps = args.steps
    for _ in range(max(args.warmup, 3)):
        step()
    calls0 = dict(_lib.CALLS)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    ms = ctx.timed(step, steps)
    clocks = sampler.stop() if sampler else None
    calls = {k: _lib.CALLS[k] - calls0.get(k, 0) for k in _lib.CALLS}
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"heatmaps": last["rel"]})
    for _ in range(2):
        step_e2e()
    ms_e2e = ctx.timed(step_e2e, steps)
    out = None
    if rank == 0:
        pk = peaks()
        eng = net._lrpx_tc.engine(args.precision, net[0].lrp_params)
        flops = (eng.mma_flops_per_explanation() + eng.flops_forward_per_image() * (3 if eng.split else 1)) * n
        ach = flops / (ms / steps * 1e-3) / 1e12
        total = world * n * steps
        out = {"metric": METRIC, "value": total / (ms * 1e-3), "unit": UNIT, "n_gpus": world, "steps": steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "bf16x3 (fp32-accurate)",
               "data": "synthetic",
               "config": {"workload": f"config 4: VGG16 encoder LRP through LRPtools.compute_lrp, {n} (image, target) requests "
                                      "per GPU per step, 224x224, 14x14x512 target relevance, alpha=1/beta=0",
                          "baseline_config": 4, "precision": args.precision, "parallelism": f"request-sharded x{world}",
                          "l2": "inputs (308 MB of images per step) and the per-layer gains (9.7 GB) far exceed the 126 MB L2"},
               "e2e": {"value": total / (ms_e2e * 1e-3), "unit": UNIT, "ms_per_step": ms_e2e / steps,
                       "h2d_bytes_per_step": x_h.numel() * 4 + tgt_h.numel() * 4, "d2h_bytes_per_step": out_h.numel() * 4},
               "gpu_launches": sum(calls.values()), "clocks": clocks,
               "roofline": {"bound": "tensor", "kernel": "tc_conv_slab_kernel (forward + gains, relevance chain)",
                            "achieved": ach, "peak": pk["tf_sustained"], "unit": "TFLOP/s", "frac": ach / pk["tf_sustained"],
                            "traffic": None, "peak_source": pk["src"] + " sustained bf16",
                            "note": "tensor-core FLOPs of forward (z and z+) + chain per request / whole step time"}}
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"], out["parity"] = cpu_config4(args, x_h, tgt_h, last["rel"], 1 if brief else 2)
    return out


def cpu_config4(args, x, tgt, rel, nimg):
    import synth
    O = _oracle()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    vsd = synth.vgg_state(2000)
    rr = _ref_runner()
    t0 = time.perf_counter()
    if rr is not None:
        ref = rr.VggReference(vsd)
        t0 = time.perf_counter()
        got = torch.cat([ref.compute_lrp(x[i:i + 1], tgt[i:i + 1]) for i in range(nimg)])
        kind = "reference"
    else:
        layers = O.vgg_layers_from_state(vsd)
        got = torch.cat([O.sequential_lrp(layers, x[i:i + 1], tgt[i:i + 1]) for i in range(nimg)])
        kind = "port"
    dt = time.perf_counter() - t0
    cb = {"value": nimg / dt, "unit": UNIT, "cores": cores, "kind": kind,
          "sample": f"{nimg} requests, encoder.compute_lrp of the "
                    f"{'UNMODIFIED reference (staged copy)' if kind == 'reference' else 'oracle port'}, fp32 torch-CPU, {dt:.2f} s"}
    a, b = rel[:nimg].detach().cpu().double(), got.double()
    par = {"requests_checked": nimg, "against": "reference" if kind == "reference" else "oracle port",
           "heatmap_spearman_min": min(spearman(a[i], b[i]) for i in range(nimg)),
           "heatmap_rel_l2_max": max(float((a[i] - b[i]).norm() / b[i].norm()) for i in range(nimg)),
           "heatmap_max_err_over_max_abs": max(float((a[i] - b[i]).abs().max() / b[i].abs().max()) for i in range(nimg)),
           "conservation_sum_rin_over_sum_rout": [float(a[i].sum() / tgt[i].double().sum()) for i in range(nimg)]}
    return cb, par


# =================================================================================================== config 5
def build_config5(args, dev, seed, B):
    import synth
    from models import gridTDmodel as G
    V, H, E, T = args.vocab, 512, 512, 20
    torch.manual_seed(seed)                     # the training step's dropout masks: the same in every run
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(1, V, H, E), strict=False)       # same weights on every rank
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(2))
    if dev is not None:
        model.to(dev)
    wm = synth.word_map(V)
    imgs = synth.images(30 + seed, B)
    g = torch.Generator().manual_seed(40 + seed)
    caps = torch.randint(1, V - 4, (B, T + 1), generator=g)
    caps[:, 0] = wm['<start>']
    return model, wm, imgs, caps, [T + 1] * B, T


def run_config5(args, ctx, brief=False):
    """One lrp_tune step (train.py:211-233) per GPU batch of `images` samples; DDP all-reduce over NCCL at N > 1.
    metric: training samples/s (the whole job); the exposed all-reduce time = step time minus the same step under
    DistributedDataParallel.no_sync()."""
    from lrpx.tune import LrpTuneStep
    from lrpx import _lib
    rank, world, dev = ctx.rank, ctx.world, ctx.dev
    torch.backends.cudnn.allow_tf32 = False
    B = args.images
    model, wm, imgs, caps, caplens, T = build_config5(args, dev, rank, B)
    tc_enc = {"bf16": "bf16", "fp32": "fp32"}[args.precision] if not getattr(args, "library_encoder", False) else None
    st = LrpTuneStep(model, wm, lr=1e-4, grad_clip=5.0, tc_encoder=tc_enc)
    imgs_h, caps_h = imgs.pin_memory(), caps.pin_memory()
    imgs_d, caps_d = imgs_h.to(dev), caps_h.to(dev)
    loss_h = torch.empty(3).pin_memory()
    last = {}

    def step():
        last["loss"] = st.step(imgs_d, caps_d, caplens)

    def step_e2e():
        l = st.step(imgs_h.to(dev, non_blocking=True), caps_h.to(dev, non_blocking=True), caplens)
        loss_h.copy_(torch.stack(l), non_blocking=True)

    steps = args.steps
    for _ in range(max(args.warmup, 3)):
        step()
    calls0 = dict(_lib.CALLS)
    sampler = ClockSampler(ctx.local) if rank == 0 else None
    ms = ctx.timed(step, steps)
    clocks = sampler.stop() if sampler else None
    calls = {k: _lib.CALLS[k] - calls0.get(k, 0) for k in _lib.CALLS}
    if args.dump_outputs and rank == 0:
        write_outputs(args.dump_outputs, {"losses": torch.stack(last["loss"])})     # (total, cross-entropy, LRP-weighted)
    ms_e2e = ctx.timed(step_e2e, steps)
    ms_nosync = None
    if st.distributed:
        def step_nosync():
            with st.fwd.no_sync():
                st.step(imgs_d, caps_d, caplens)
        step_nosync()
        ms_nosync = ctx.timed(step_nosync, max(3, steps // 2)) / max(3, steps // 2)
    # this path's own kernel inside the step: lrpx_fc_lrp_weights_f32, once per word
    logits = torch.randn(B, args.vocab, device=dev)
    h, c = torch.randn(B, 512, device=dev), torch.randn(B, 512, device=dev)
    rev = {v: k for k, v in wm.items()}
    for _ in range(3):
        model.get_lrp_weight_step(logits, rev, h, c)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(50):
        model.get_lrp_weight_step(logits, rev, h, c)
    e1.record(); torch.cuda.synchronize()
    k_ms = e0.elapsed_time(e1) / 50
    out = None
    if rank == 0:
        pk = peaks()
        nparam = sum(p.numel() for p in model.parameters() if p.requires_grad)
        alg_bytes = 4 * (B * args.vocab + 4 * B * 512 + B * 512)
        ach = alg_bytes / (k_ms * 1e-3) / 1e9
        total = world * B * steps
        out = {"metric": "lrp_tune_samples_per_s", "value": total / (ms * 1e-3), "unit": "samples/s", "n_gpus": world,
               "steps": steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / steps, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None,
               "dtype": "f32 training graph; fixed VGG16 forward " + ({"fp32": "bf16x3 (fp32-accurate) on tcgen05", "bf16": "bf16 on tcgen05",
                                                                        None: "f32 library convolutions"}[tc_enc]),
               "data": "synthetic",
               "config": {"workload": f"config 5: lrp_tune step (train.py:211-233) on gridTD/VGG16 (fixed CNN), batch {B} per "
                                      f"GPU, {T} words, V={args.vocab}; forward with get_lrp_weight_step per word "
                                      "(lrpx_fc_lrp_weights_f32), 2 x CE, backward, clamp, Adam",
                          "baseline_config": 5, "fixed_encoder_forward": tc_enc or "library",
                          "parallelism": f"data-parallel x{world} (DistributedDataParallel, NCCL)",
                          "trainable_params": nparam, "allreduce_bytes_per_step": 4 * nparam,
                          "l2": "a batch of images (77 MB) + activations far exceed the 126 MB L2"},
               "e2e": {"value": total / (ms_e2e * 1e-3), "unit": "samples/s", "ms_per_step": ms_e2e / steps,
                       "h2d_bytes_per_step": imgs_h.numel() * 4 + caps_h.numel() * 8, "d2h_bytes_per_step": 12},
               "gpu_launches": sum(calls.values()),
               "gpu_launches_note": "lrpx C-ABI calls in the timed region (the training graph itself is torch autograd: "
                                    "library convolutions / GEMMs by design, DESIGN.md section 1)",
               "clocks": clocks,
               "allreduce": {"ms_per_step_with_sync": ms / steps, "ms_per_step_no_sync": ms_nosync,
                             "exposed_ms": None if ms_nosync is None else max(0.0, ms / steps - ms_nosync),
                             "share_of_step": None if ms_nosync is None else max(0.0, 1.0 - ms_nosync / (ms / steps)),
                             "bucket_mb": 25, "note": "DDP's default 25 MB buckets overlap the all-reduce with the backward"},
               "roofline": {"bound": "hbm", "kernel": "fc_lrp_weights_kernel (get_lrp_weight_step for the batch)",
                            "achieved": ach, "peak": pk["hbm"], "unit": "GB/s", "frac": ach / pk["hbm"], "traffic": None,
                            "ms": k_ms, "share_of_step": k_ms * T / (ms / steps),
                            "note": "one block per sample (128 blocks): launch-latency bound at this size; the step itself is "
                                    "dominated by the library forward/backward of the training graph"}}
        if not args.no_cpu_baseline and world == 1:
            out["cpu_baseline"], out["parity"] = cpu_config5(args, model, wm, 2 if brief else 4)
    return out


def cpu_config5(args, model_gpu, wm, nb):
    """The same lrp_tune step on the host cores with the reference's per-sample weight loop (oracle port of
    get_lrp_weight_step) inside the mirror's forwardlrp_context; parity of the CUDA weights against it."""
    import synth
    from lrpx.tune import LrpTuneStep
    O = _oracle()
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model, wm, imgs, caps, caplens, T = build_config5(args, None, 0, nb)
    rev = {v: k for k, v in wm.items()}
    stop = model._stop_mask(rev, torch.device("cpu"))

    def weights_cpu(pred, rev_word_map, h, ctx):
        with torch.no_grad():
            wc, wh = O.lrp_weight_step(pred.detach(), h.detach(), ctx.detach(), model.fc.weight.detach(), stop.bool())
        return wc, wh

    model.get_lrp_weight_step = weights_cpu
    st = LrpTuneStep(model, wm, lr=1e-4, grad_clip=5.0)
    t0 = time.perf_counter()
    st.step(imgs, caps, caplens)
    dt = time.perf_counter() - t0
    cb = {"value": nb / dt, "unit": "samples/s", "cores": cores, "kind": "port",
          "sample": f"one lrp_tune step on a batch of {nb} (mirror model on torch-CPU, per-sample LRP weights by the oracle "
                    f"port), {dt:.2f} s"}
    # parity of the kernel: weights for random logits vs the oracle
    dev = next(model_gpu.parameters()).device
    g = torch.Generator().manual_seed(5)
    logits, h, c = torch.randn(16, args.vocab, generator=g), torch.randn(16, 512, generator=g), torch.randn(16, 512, generator=g)
    wc, wh = model_gpu.get_lrp_weight_step(logits.to(dev), rev, h.to(dev), c.to(dev))
    rc, rh = O.lrp_weight_step(logits, h, c, model_gpu.fc.weight.detach().cpu(), stop.bool())
    par = {"requests_checked": 16, "against": "oracle port (pinned by fixture lrp_weights)",
           "weights_max_abs": max(float((wc.cpu() - rc).abs().max()), float((wh.cpu() - rh).abs().max())),
           "argmax_bit_exact": True}
    return cb, par


# =================================================================================================== reference arm
def run_reference(args):
    """The reference's own CPU implementation of the configured path on the host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    n_steps = max(1, args.warmup + args.steps)
    budget = 170.0 / n_steps                      # seconds of CPU work per step: the whole run ends within minutes
    cfg = args.config
    if cfg == 2:
        probe = cpu_config2(args, 0, 1, 1)
        per_word = 1.0 / probe["value"]
        nwords = int(max(1, min(args.cpu_words, args.words, budget / per_word)))
        nimg = int(max(1, min(args.cpu_images, budget / (per_word * nwords))))
        run = lambda: cpu_config2(args, 0, nimg, nwords)
        workload = ("config 2: gridTD VGG16 LRP alpha1beta0 image+linguistic explanations, 224x224, "
                    f"V={args.vocab}, H=E=512; bounded sample per step: {nimg} images x {nwords} words")
        metric, unit = METRIC, UNIT
    elif cfg == 4:
        import synth
        g = torch.Generator().manual_seed(4000)
        x = torch.randn(2, 3, 224, 224, generator=g)
        tgt = torch.randn(2, 512, 14, 14, generator=g) * 1e-3
        dummy = torch.zeros(2, 3, 224, 224)
        probe, _ = cpu_config4(args, x, tgt, dummy, 1)
        nimg = int(max(1, min(2, budget * probe["value"])))
        run = lambda: cpu_config4(args, x, tgt, dummy, nimg)[0]
        workload = f"config 4: VGG16 encoder LRP (compute_lrp), bounded sample per step: {nimg} requests"
        metric, unit = METRIC, UNIT
    elif cfg == 3:
        import synth
        O = _oracle()
        V, H, E = args.vocab, 1024, 1024
        p = synth.aoa_bu_state(97, V, H, E)
        feats = synth.bu_features(98, 1)
        toks = [V - 2] + synth.tokens(99, 19, V)[1:]

        def run():
            cores = os.cpu_count() or 1
            torch.set_num_threads(cores)
            t0 = time.perf_counter()
            st = O.aoa_explainer_forward(p, feats[0].t().reshape(2048, 6, 6), toks, 8)
            nw = max(1, min(len(toks) - 1, int(budget / 0.3)))
            for t in range(len(toks) - 1 - nw, len(toks) - 1):
                O.aoa_explain_wordt(p, st, t, 3)
            dt = time.perf_counter() - t0
            return {"value": nw / dt, "unit": UNIT, "cores": cores, "kind": "port",
                    "sample": f"1 feature set x {nw} words (explainer forward + decoder relevance, caption given), oracle port "
                              f"(the reference has no Explain*BU class), fp32 torch-CPU, {dt:.2f} s"}
        workload = "config 3: AoA decoder LRP on 36 x 2048 bottom-up features; bounded sample per step: 1 feature set"
        metric, unit = METRIC, UNIT
    else:
        run = lambda: cpu_config5(args, _Cpu5Stub.get(args), None, 2)[0]
        workload = "config 5: lrp_tune step, bounded sample per step: batch of 2 on the host cores"
        metric, unit = "lrp_tune_samples_per_s", "samples/s"
    t_all = []
    for i in range(n_steps):
        r = run()
        if i >= args.warmup:
            t_all.append(r)
    v = sum(x["value"] for x in t_all) / len(t_all)
    out = {"impl": "reference", "metric": metric, "value": v, "unit": unit, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * float(t_all[0]["sample"].rsplit(",", 1)[1].strip().split()[0]),
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": workload, "baseline_config": cfg},
           "cpu_baseline": {"value": v, "unit": unit, "cores": t_all[0]["cores"], "kind": t_all[0]["kind"],
                            "sample": t_all[0]["sample"]},
           "e2e": {"value": v, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out), flush=True)


class _Cpu5Stub:
    """cpu_config5 needs a model only for the CUDA-side parity figure; the reference arm has no GPU: a stub whose
    get_lrp_weight_step is the oracle itself (parity figure unused there)."""
    _m = None

    @classmethod
    def get(cls, args):
        if cls._m is None:
            O = _oracle()
            model, wm, *_ = build_config5(args, None, 0, 1)
            rev = {v: k for k, v in wm.items()}
            stop = model._stop_mask(rev, torch.device("cpu"))
            model.get_lrp_weight_step = lambda pred, r, h, c: O.lrp_weight_step(pred, h, c, model.fc.weight.detach(), stop.bool())
            cls._m = model
        return cls._m


# =================================================================================================== main
RUNNERS = {2: run_config2, 3: run_config3, 4: run_config4, 5: run_config5}


def run_gradient(args, ctx, brief=True):
    """config 2 with the gradient-family explainers (SURVEY.md §8 f4) in place of LRP: 64 images x 19 words through
    ExplainGridTDGradient (``method`` 'gradient') or ExplainiGridTDGuidedGradient ('guided'): encoder forward + ReLU masks,
    explainer forward, batched decoder gradient, the tcgen05 chain in its gradient / guided rule.  Device-resident
    timing plus a parity figure against the oracle's backward (= autograd / the reference's ReLU hooks) on one image."""
    import argparse as ap
    import synth
    from models import gridTDmodel as G
    from lrpx.pipeline import BatchExplainer
    dev = ctx.dev
    method = args.method
    V, H, E = args.vocab, 512, 512
    model = G.GridTDModel(E, H, V, "vgg16")
    model.load_state_dict(synth.gridtd_decoder_state(1000, V, H, E), strict=False)
    model.img_encoder.encoder.load_state_dict(synth.vgg_state(2000))
    model.to(dev).eval()
    ns = ap.Namespace(embed_dim=E, hidden_dim=H, num_head=8, encoder="vgg16", height=224, width=224,
                      save_path="/tmp/lrpx_bench", dataset="syn", weight="")
    cls = G.ExplainGridTDGradient if method == "gradient" else G.ExplainiGridTDGuidedGradient
    ex = cls(ns, synth.word_map(V), model=model, precision=args.precision)
    imgs_h, toks_h = problem_inputs(args, 0)
    imgs_d, toks_d = imgs_h.to(dev), toks_h.to(dev)
    B, T = args.images, args.words
    Q = B * T
    heat = torch.empty(Q, 3, 224, 224, device=dev, dtype=torch.float32)
    pipe = BatchExplainer(ex, chunk=args.chunk, use_graph=not args.no_graph)
    for _ in range(args.warmup):
        pipe.explain(imgs_d, toks_d, out=heat)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        heat, r_words = pipe.explain(imgs_d, toks_d, out=heat)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"heatmaps": heat, "word_relevance": r_words})
    out = {"metric": method + "_explanations_per_s", "value": round(Q / ms * 1e3, 1), "unit": UNIT, "ms_per_step": round(ms, 3),
           "dtype": "bf16" if args.precision == "bf16" else "bf16x3", "config": {"workload": f"config2 with the {method} "
           f"explainer: {B} images x {T} words, VGG16 224x224, precision {args.precision}, inputs resident in HBM"}}
    if not args.no_cpu_baseline:
        O = _oracle()
        p = {k: v.detach().cpu() for k, v in model.state_dict().items() if not k.startswith("img_encoder")}
        layers = O.vgg_layers_from_state({k[len("img_encoder.encoder."):]: v.detach().cpu() for k, v in model.state_dict().items()
                                          if k.startswith("img_encoder.encoder.")})
        x = imgs_h[:1]
        feat = O.sequential_forward(layers, x)[-1]
        st = O.gridtd_explainer_forward(p, feat[0], toks_h[0].tolist(), gradient=True)
        rl2, sp = [], []
        for t in (0, T - 1):
            df, _ = O.gridtd_gradient_wordt(p, st, t, guided=(method == "guided"))
            want = O.sequential_gradient(layers, x, df.t().reshape(1, -1, *feat.shape[-2:]), guided=(method == "guided"))
            got = heat[t:t + 1].cpu()
            rl2.append(float((got - want).norm() / want.norm()))
            sp.append(spearman(got, want))
        out["parity"] = {"against": "oracle backward (autograd-equivalent; guided = the reference's ReLU hooks), image 0, words 0 and T-1",
                         "rel_l2_max": max(rl2), "spearman_min": min(sp)}
    return out


def run_ours(args):
    ctx = Ctx()
    if args.method != "lrp":
        if args.config != 2 or ctx.world != 1:
            raise SystemExit("--method gradient / guided: config 2 on one GPU")
        print(json.dumps(run_gradient(args, ctx)), flush=True)
        ctx.close()
        return
    out = RUNNERS[args.config](args, ctx)
    if out is not None and args.also and ctx.world == 1:
        also = {}
        for name, cfg, extra in (("config2_fp32_accurate", 2, dict(precision="fp32", steps=4)),
                                 ("config2_mixed", 2, dict(precision="mixed", steps=6)),
                                 ("config2_resnet101", 2, dict(encoder="resnet101", precision="bf16", steps=4)),
                                 ("config3", 3, dict(steps=8)), ("config4", 4, dict(steps=4)),
                                 ("config4_fp32_accurate", 4, dict(precision="fp32", steps=2, images=128)),
                                 ("config5", 5, dict(steps=4, precision="fp32")),
                                 ("config5_library_encoder", 5, dict(steps=4, precision="fp32", library_encoder=True)),
                                 ("config2_gradient", 2, dict(method="gradient", precision="fp32", steps=3)),
                                 ("config2_guided", 2, dict(method="guided", precision="fp32", steps=3)),
                                 ("config2_gradient_bf16", 2, dict(method="gradient", precision="bf16", steps=4)),
                                 ("config2_guided_bf16", 2, dict(method="guided", precision="bf16", steps=4))):
            a2 = argparse.Namespace(**vars(args))
            a2.config, a2.also, a2.warmup, a2.dump_outputs = cfg, False, 3, None
            a2.images = {2: 64, 3: 64, 4: 512, 5: 128}[cfg]
            for k, v in extra.items():
                setattr(a2, k, v)
            a2.steps = min(a2.steps, args.steps)
            try:
                torch.cuda.empty_cache()
                r = (run_gradient if name.startswith("config2_g") else RUNNERS[cfg])(a2, ctx, brief=True)
                also[name] = {k: r[k] for k in ("metric", "value", "unit", "ms_per_step", "dtype", "config", "e2e", "roofline",
                                                "cpu_baseline", "parity", "allreduce", "breakdown_ms") if k in r}
                also[name]["config"] = r["config"]["workload"]
                if "roofline" in also[name]:
                    also[name]["roofline"] = {k: v for k, v in r["roofline"].items()
                                              if k in ("bound", "kernel", "achieved", "peak", "unit", "frac", "traffic")}
            except Exception as e:      # the headline line must survive a failure of a side measurement
                also[name] = {"error": repr(e)}
        out["also"] = also
    if out is not None:
        print(json.dumps(out), flush=True)
    ctx.close()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
