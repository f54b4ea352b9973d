"""Cost of the class count: the graph-replayed DA step and the full-resolution evaluation at several counts.

    python scripts/bench_classes.py [--counts 13,16,19,32] [--out profiles/r3_bench_classes.json]

Per class count n:
* DA step: BiSeNet("STDCNet813", n) + FCDiscriminator(n), optim.FusedSGD / FusedAdam, 8 source + 8 target
  images of 512x1024 (bench.py's da_dense workload), the whole step replayed as one CUDA graph.  CUDA
  events around --steps replays, --repeats times after --warmup replays: ms per step of every repeat.
* eval: train.val over 8 images of 1024x2048 (bench.py's eval workload, eager: val ends in a host read).
* up-sampling kernels: torch.profiler over --prof-steps EAGER DA steps (a separate pass, after the timed
  ones): device time per step of every csrc/loss.cu up-sampling kernel, and of the whole step.
The card's name, power limit and maximum SM clock are read in the same run (nvidia-smi query)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dasemanticsegmentationaml_b200 import optim as B200Optim  # noqa: E402
from dasemanticsegmentationaml_b200 import train as T  # noqa: E402
from dasemanticsegmentationaml_b200.model import BiSeNet, FCDiscriminator  # noqa: E402


def card():
    dev = torch.cuda.current_device()
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm",
                            "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=30)
        pl, clk = [v.strip() for v in r.stdout.strip().split(",")]
        info.update(power_limit_w=float(pl), sm_clock_max_mhz=float(clk))
    except Exception as ex:  # the numbers are still reported, without the power limit
        info["power_limit_w"] = "unavailable (%r)" % (ex,)
    return info


def spread(vals):
    return {"median": statistics.median(vals), "min": min(vals), "max": max(vals), "repeats": vals}


def time_calls(fn, steps, repeats, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / steps)
    return out


def data(n_classes, batch, h, w, seed, target=True):
    g = torch.Generator().manual_seed(seed)
    labels = torch.randint(0, n_classes + 1, (batch, h, w), generator=g)
    labels[labels == n_classes] = 255
    d = {"images": torch.randn(batch, 3, h, w, generator=g), "labels": labels}
    if target:
        d["images_t"] = torch.randn(batch, 3, h, w, generator=g)
    return {k: v.cuda() for k, v in d.items()}


def upsample_profile(step, n_steps):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_steps):
            step()
        torch.cuda.synchronize()
    per_kernel, total = {}, 0.0
    for ev in prof.events():
        if ev.device_type != torch.autograd.DeviceType.CUDA:
            continue
        us = ev.device_time if hasattr(ev, "device_time") else ev.cuda_time
        total += us
        if "upsample_" in ev.name:
            name = ev.name.split("(")[0].replace("void b200::", "")
            per_kernel[name] = per_kernel.get(name, 0.0) + us
    per_kernel = {k: round(v / n_steps, 1) for k, v in sorted(per_kernel.items())}
    return {"us_per_step": per_kernel, "upsample_us_per_step": round(sum(per_kernel.values()), 1),
            "all_kernels_us_per_step": round(total / n_steps, 1)}


def run_count(n_classes, args):
    torch.manual_seed(0)
    model = BiSeNet("STDCNet813", n_classes).cuda()
    disc = FCDiscriminator(n_classes).cuda()
    opt = B200Optim.FusedSGD(model.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
    opt_d = B200Optim.FusedAdam(disc.parameters(), lr=1e-3, betas=(0.9, 0.99))
    buf = data(n_classes, 8, 512, 1024, seed=100)

    def eager(images, labels, images_t):
        return T.train_da_step(model, disc, opt, opt_d, images, labels, images_t)

    graphed = T.GraphedStep(eager, buf, optimizers=[opt, opt_d])
    da = time_calls(graphed, args.steps, args.repeats, args.warmup)
    losses = [float(v) for v in graphed()]

    ev = data(n_classes, 8, 1024, 2048, seed=200, target=False)
    batches = [(ev["images"], ev["labels"])]
    res = {}
    ev_ms = time_calls(lambda: res.update(v=T.val(model, batches)), args.eval_steps, args.repeats, 2)
    prof = upsample_profile(lambda: eager(**buf), args.prof_steps)
    del graphed
    return {"da_step_ms": spread(da), "da_img_per_s": round(16 / (statistics.median(da) * 1e-3), 1),
            "last_losses": losses, "eval_ms": spread(ev_ms),
            "eval_img_per_s": round(8 / (statistics.median(ev_ms) * 1e-3), 1), "miou": res["v"][1],
            "upsample_kernels_eager_da_step": prof}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--counts", default="13,16,19,32")
    ap.add_argument("--steps", type=int, default=20, help="graph replays per timed repeat")
    ap.add_argument("--eval-steps", type=int, default=5, help="evaluations per timed repeat")
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--prof-steps", type=int, default=3)
    ap.add_argument("--out", default=None, help="write the JSON result here (default: stdout only)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_classes.py measures on the GPU; no CUDA device found")
    result = {"card": card(), "torch": torch.__version__, "time": time.strftime("%Y-%m-%d %H:%M:%S"),
              "da_step": "BiSeNet STDCNet813 + FCDiscriminator, 8 + 8 images of 512x1024, graph replay",
              "eval": "train.val, 8 images of 1024x2048, eager", "args": vars(args), "counts": {}}
    for n in [int(v) for v in args.counts.split(",")]:
        result["counts"][str(n)] = run_count(n, args)
        r = result["counts"][str(n)]
        print("n=%2d  DA step %.3f ms [%.3f, %.3f]  eval %.2f ms  up-sampling %.1f us/step (eager)"
              % (n, r["da_step_ms"]["median"], r["da_step_ms"]["min"], r["da_step_ms"]["max"], r["eval_ms"]["median"],
                 r["upsample_kernels_eager_da_step"]["upsample_us_per_step"]), flush=True)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
