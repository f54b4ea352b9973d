"""Cost of multi-scale + flip evaluation (train.predict) at the Cityscapes evaluation size.

    python scripts/bench_tta.py [--repeats 20] [--out profiles/bench_tta.json]

BiSeNet("STDCNet813", 19) in eval mode, 8 images of 1024x2048 (bench.py's eval workload), three configurations:
single scale (the existing path), flip only, and scales (0.5, 0.75, 1.0, 1.25, 1.5, 1.75) with flip.
* predict: CUDA events around each whole call, --repeats times after --warmup calls.
* image_rescale: every scale's launch (with mirrors) alone; achieved GB/s on the algorithmic bytes (source read
  once, outputs written once), against the HBM rate bench.py's roofline_mem uses.
* msc_argmax: the six-scale + flip combine (12 maps) alone, on the maps of a real forward; ns per output pixel
  per map, and its share of the predict time.
All working sets exceed the 126 MB L2 except the combine's maps at the smallest scales.  Every shape is warmed
up first.  A prediction check runs the largest forward of the benchmark (2N = 16 images of 1792x3584,
scales=(1.75,) with flip) and compares image 0 with the fp32 oracle's MscEval.  The card's name, power limit
and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from bench import measured_peaks  # noqa: E402
from dasemanticsegmentationaml_b200 import kernels as K  # noqa: E402
from dasemanticsegmentationaml_b200 import train as T  # noqa: E402
from dasemanticsegmentationaml_b200.model import BiSeNet  # noqa: E402
from scripts.bench_classes import card  # noqa: E402

SCALES6 = (0.5, 0.75, 1.0, 1.25, 1.5, 1.75)
CONFIGS = {"single": ((1.0,), False), "flip": ((1.0,), True), "6scales_flip": (SCALES6, True)}


def spread(vals):
    return {"median": round(statistics.median(vals), 4), "min": round(min(vals), 4), "max": round(max(vals), 4),
            "repeats": len(vals)}


def time_each(fn, repeats, warmup):
    """ms of every call, CUDA events around each one."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1))
    return out


def prediction_check(model, x):
    """scales=(1.75,) with flip over all images (one forward of 2N images of 1792x3584), image 0 against the
    fp32 oracle."""
    from oracle import segnet_oracle as O
    from tests.helpers import to_device
    from tests.test_tta_gpu import msc_predict
    pred = T.predict(model, x, scales=(1.75,), flip=True)
    sd = to_device(O.make_bisenet_state(seed=0), "cuda")
    with torch.no_grad():
        ref, _ = msc_predict(sd, x[:1], 19, (1.75,), True)
    agree = (pred[:1].long() == ref).double().mean().item()
    return {"scales": [1.75], "flip": True, "forward_images": 2 * x.shape[0], "forward_size": [1792, 3584],
            "argmax_agreement_image0": round(agree, 6), "gate": 0.995, "passed": agree >= 0.995}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the JSON result here (default: stdout only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_tta.py measures on the GPU; no CUDA device found")
    from tests.helpers import load_oracle_state
    from oracle import segnet_oracle as O
    model = load_oracle_state(BiSeNet("STDCNet813", 19), O.make_bisenet_state(seed=0)).cuda().eval()
    x = torch.randn(8, 3, 1024, 2048, generator=torch.Generator().manual_seed(0)).cuda()
    N, _, H, W = x.shape
    peaks = measured_peaks()
    result = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%d %H:%M:%S"),
              "workload": "BiSeNet STDCNet813, 19 classes, eval, 8 images of 1024x2048", "args": vars(args),
              "hbm_gbs_reference": {"gbs": peaks["hbm"], "source": peaks["source"]}}

    pred = {}
    for name, (scales, flip) in CONFIGS.items():
        ms = time_each(lambda: T.predict(model, x, scales=scales, flip=flip), args.repeats, args.warmup)
        pred[name] = {"scales": list(scales), "flip": flip, "maps": len(scales) * (2 if flip else 1), "ms": spread(ms)}
        print("predict %-13s %8.2f ms [%.2f, %.2f]" % (name, statistics.median(ms), min(ms), max(ms)), flush=True)
    result["predict"] = pred

    resc = {}
    for s in SCALES6:
        h, w = int(s * H), int(s * W)
        dst = torch.empty((2 * N, 3, h, w), dtype=torch.float32, device="cuda")
        ms = time_each(lambda: K.image_rescale(x, dst, mirror=True), args.repeats, args.warmup)
        nbytes = 4.0 * (x.numel() + dst.numel())
        gbs = nbytes / (statistics.median(ms) * 1e-3) / 1e9
        resc[str(s)] = {"out": [2 * N, 3, h, w], "ms": spread(ms), "mbytes": round(nbytes / 1e6, 1),
                        "gbs": round(gbs, 1), "frac_of_hbm": round(gbs / peaks["hbm"], 3)}
        print("image_rescale %.2f -> %dx%d x2: %.3f ms  %.0f GB/s (%.2f of HBM)"
              % (s, h, w, statistics.median(ms), gbs, gbs / peaks["hbm"]), flush=True)
        del dst
    result["image_rescale"] = resc

    # the six-scale + flip combine on the maps of a real forward (the loop of train.predict)
    maps, mirrored = [], []
    with torch.no_grad():
        for s in SCALES6:
            xs = torch.empty((2 * N, 3, int(s * H), int(s * W)), dtype=torch.float32, device="cuda")
            K.image_rescale(x, xs, mirror=True)
            lr = model.forward_lowres(xs)[0]
            maps += [lr[:N], lr[N:]]
            mirrored += [False, True]
            del xs
    out = torch.empty((N, H, W), dtype=torch.uint8, device="cuda")
    ms = time_each(lambda: K.msc_argmax(maps, mirrored, H, W, 19, out), args.repeats, args.warmup)
    med = statistics.median(ms)
    total = pred["6scales_flip"]["ms"]["median"]
    result["msc_argmax"] = {"maps": len(maps), "ms": spread(ms),
                            "ns_per_pixel_map": round(med * 1e6 / (N * H * W * len(maps)), 4),
                            "share_of_predict_6scales_flip": round(med / total, 4),
                            "maps_mbytes": round(sum(m.numel() * 4 for m in maps) / 1e6, 1)}
    print("msc_argmax 12 maps: %.3f ms  %.4f ns per pixel-map  %.1f%% of predict"
          % (med, result["msc_argmax"]["ns_per_pixel_map"], 100 * med / total), flush=True)
    del maps, lr
    torch.cuda.empty_cache()

    result["prediction_check"] = prediction_check(model, x)
    print("prediction check:", result["prediction_check"], flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)
    if not result["prediction_check"]["passed"]:
        sys.exit("prediction check failed")


if __name__ == "__main__":
    main()
