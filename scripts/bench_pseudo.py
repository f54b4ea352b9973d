"""Cost of the pseudo-label round (train.predict_confidence, pseudo_label_thresholds, pseudo_labels).

    python scripts/bench_pseudo.py [--repeats 10] [--out profiles/bench_pseudo.json]

(a) predict_confidence against predict: BiSeNet("STDCNet813", 19) in eval mode, 8 images of 1024x2048, at one
    scale and at scales (0.5, 0.75, 1.0, 1.25, 1.5, 1.75) with flip.  CUDA events around each whole call, the
    two functions alternated call by call so that both see the same clocks.
(b) pseudo_label_thresholds over 372 seeded batches of 8 x 512 x 1024 uint8 predictions (19 classes, uniform)
    and fp32 confidences (2976 images, Cityscapes train's size: 1.56 G pixels, 7.8 GB), no model needed; conf
    uniform in (1/19, 1] and concentrated near 1 (1 - 0.1 u^3).  The whole call, and each pass's histogram
    launches alone (CUDA events around the 372 launches of one pass); achieved GB/s on 5 bytes per pixel
    against the HBM rate bench.py uses.  The set is 60x the 126 MB L2, so every pass reads HBM.
(c) pseudo_labels over the same set with uint8 and int64 output, GB/s on 5 + 1 or 5 + 8 bytes per pixel.
The card's name, power limit and maximum SM clock are read in the same run."""
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
from scripts.bench_tta import SCALES6, spread  # noqa: E402

N_BATCHES, BATCH = 372, (8, 512, 1024)


def event_ms(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def bench_predict(args):
    from oracle import segnet_oracle as O
    from tests.helpers import load_oracle_state
    model = load_oracle_state(BiSeNet("STDCNet813", 19), O.make_bisenet_state(seed=0)).cuda().eval()
    x = torch.randn(8, 3, 1024, 2048, generator=torch.Generator().manual_seed(0)).cuda()
    out = {}
    for name, (scales, flip) in {"single": ((1.0,), False), "6scales_flip": (SCALES6, True)}.items():
        fns = {"predict": lambda: T.predict(model, x, scales=scales, flip=flip),
               "predict_confidence": lambda: T.predict_confidence(model, x, scales=scales, flip=flip)}
        for fn in fns.values():
            for _ in range(args.warmup):
                fn()
        ms = {k: [] for k in fns}
        for _ in range(args.repeats):
            for k, fn in fns.items():
                ms[k].append(event_ms(fn))
        a, b = statistics.median(ms["predict"]), statistics.median(ms["predict_confidence"])
        out[name] = {"scales": list(scales), "flip": flip, "predict_ms": spread(ms["predict"]),
                     "predict_confidence_ms": spread(ms["predict_confidence"]), "ratio": round(b / a, 4)}
        print("%-13s predict %8.2f ms  predict_confidence %8.2f ms  ratio %.3f" % (name, a, b, b / a), flush=True)
    del model, x
    torch.cuda.empty_cache()
    return out


def target_set(kind, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    preds, confs = [], []
    for _ in range(N_BATCHES):
        preds.append(torch.randint(0, 19, BATCH, device="cuda", generator=g, dtype=torch.uint8))
        u = torch.rand(BATCH, device="cuda", generator=g)
        confs.append(1.0 - (1.0 - 1.0 / 19) * u if kind == "uniform" else 1.0 - 0.1 * u ** 3)
    return preds, confs


def bench_select(args, hbm):
    out = {}
    px = N_BATCHES * BATCH[0] * BATCH[1] * BATCH[2]
    for kind in ("uniform", "concentrated"):
        preds, confs = target_set(kind, seed=1 if kind == "uniform" else 2)
        T.pseudo_label_thresholds(preds, confs, 19)     # warm-up
        torch.cuda.synchronize()
        whole = [event_ms(lambda: T.pseudo_label_thresholds(preds, confs, 19)) for _ in range(args.repeats)]
        n = 19
        state = torch.empty(3 * n, dtype=torch.int64, device="cuda")
        hist = torch.zeros(n * 256, dtype=torch.int64, device="cuda")
        thr = torch.empty(n, device="cuda")
        counts = torch.empty(n, dtype=torch.int64, device="cuda")
        passes = {p: [] for p in range(4)}
        for _ in range(args.repeats):
            for p in range(4):
                passes[p].append(event_ms(lambda: [K.class_select_hist(a, b, n, p, state, hist)
                                                   for a, b in zip(preds, confs)]))
                K.class_select_pick(n, p, 0.5, 0.9, state, hist, thr, counts)
        per = {}
        for p, ms in passes.items():
            gbs = 5.0 * px / (statistics.median(ms) * 1e-3) / 1e9
            per["pass%d" % p] = {"ms": spread(ms), "gbs": round(gbs, 1), "frac_of_hbm": round(gbs / hbm, 3)}
            print("%-12s hist pass %d: %8.2f ms  %7.0f GB/s  %.2f of HBM"
                  % (kind, p, statistics.median(ms), gbs, gbs / hbm), flush=True)
        med = statistics.median(whole)
        out[kind] = {"pixels": px, "mbytes": round(5.0 * px / 1e6, 1), "thresholds_ms": spread(whole),
                     "thresholds_gbs_4_passes": round(4 * 5.0 * px / (med * 1e-3) / 1e9, 1), "hist_passes": per,
                     "thr_portion0.5_cap0.9": [round(v, 6) for v in thr.tolist()]}
        print("%-12s pseudo_label_thresholds: %8.2f ms (4 passes + picks)" % (kind, med), flush=True)
        if kind == "concentrated":
            thr_t, _ = T.pseudo_label_thresholds(preds, confs, 19)
            app = {}
            for dtype in (torch.uint8, torch.int64):
                # one batch at a time, freed at once: the int64 labels of the whole set would be 12.5 GB
                ms = []
                for _ in range(args.repeats):
                    e = 0.0
                    for a, b in zip(preds, confs):
                        e += event_ms(lambda: T.pseudo_labels(a, b, thr_t, dtype=dtype))
                    ms.append(e)
                nbytes = px * (5.0 + torch.empty((), dtype=dtype).element_size())
                gbs = nbytes / (statistics.median(ms) * 1e-3) / 1e9
                app[str(dtype).replace("torch.", "")] = {"ms": spread(ms), "gbs": round(gbs, 1),
                                                         "frac_of_hbm": round(gbs / hbm, 3)}
                print("pseudo_labels %s: %8.2f ms  %7.0f GB/s  %.2f of HBM"
                      % (dtype, statistics.median(ms), gbs, gbs / hbm), flush=True)
            out["apply"] = app
        del preds, confs
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="write the JSON result here (default: stdout only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_pseudo.py measures on the GPU; no CUDA device found")
    peaks = measured_peaks()
    result = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%d %H:%M:%S"),
              "args": vars(args), "hbm_gbs_reference": {"gbs": peaks["hbm"], "source": peaks["source"]}}
    result["predict"] = bench_predict(args)
    result["select"] = bench_select(args, peaks["hbm"])
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
