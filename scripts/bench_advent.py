"""Cost of ADVENT's steps (train.train_minent_step, train.train_advent_step) and of csrc/entropy.cu's kernels.

    python scripts/bench_advent.py [--repeats 5] [--replays 20] [--out profiles/bench_advent.json]

(a) Graph-replayed steps: BiSeNet("STDCNet813", 19) + FCDiscriminator(19), optim.FusedSGD / FusedAdam, 8 source
    + 8 target images of 512x1024.  MinEnt, AdvEnt and train_da_step are each captured once; then, per repeat,
    each is replayed `--replays` times between CUDA events, the three alternated so that they see the same
    clocks.  Median ms per step over the repeats, with min and max.
(b) Kernels at the step's shape (8 x 64x128 logits -> 512x1024, 19 classes), each against the existing kernel
    it parallels, alternated in the same session, CUDA events around 50 launches:
      entropy training pass (b200_entropy_bwd mode 0)   vs  the CE training pass (b200_upsample_bwd mode 1)
      self-information forward (entropy_fwd mode 1, zero-bordered) vs the softmax forward (upsample_fwd mode 2)
      self-information backward (entropy_bwd mode 1, zero-bordered) vs the softmax backward (upsample_bwd mode 2)
      entropy forward without a map (entropy_fwd mode 0)
    The bf16 maps are 2.2x the 126 MB L2 together with the logits, so their traffic goes to HBM.
(c) GB/s on algorithmic bytes for the map modes: logits read once (fp32, 32 floats per pixel) plus the map
    (bf16, 32 channels) written or read, plus d_lr read and written in the backward.
The card's name, power limit and maximum SM clock are read in the same run."""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dasemanticsegmentationaml_b200 import kernels as K  # noqa: E402
from dasemanticsegmentationaml_b200 import optim as B200Optim  # noqa: E402
from dasemanticsegmentationaml_b200 import train as T  # noqa: E402
from dasemanticsegmentationaml_b200.model import BiSeNet, FCDiscriminator  # noqa: E402
from scripts.bench_classes import card  # noqa: E402

N, H, W, NCLS = 8, 512, 1024, 19


def spread(vals):
    return {"median": round(statistics.median(vals), 4), "min": round(min(vals), 4), "max": round(max(vals), 4),
            "repeats": len(vals)}


def bench_steps(args):
    from oracle import segnet_oracle as O
    from tests.helpers import load_oracle_state
    g = torch.Generator().manual_seed(0)
    x = torch.randn(N, 3, H, W, generator=g).cuda()
    xt = torch.randn(N, 3, H, W, generator=g).cuda()
    labels = torch.randint(0, NCLS, (N, H, W), generator=g).cuda()
    graphs = {}
    for name in ("minent", "advent", "da_step"):
        m = load_oracle_state(BiSeNet("STDCNet813", NCLS), O.make_bisenet_state(seed=0)).cuda()
        d = load_oracle_state(FCDiscriminator(NCLS), O.make_discriminator_state("dense", seed=4)).cuda()
        opt = B200Optim.FusedSGD(m.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
        opt_d = B200Optim.FusedAdam(d.parameters(), lr=1e-4, betas=(0.9, 0.99))
        if name == "minent":
            def fn(images, labels, images_t, m=m, opt=opt):
                return T.train_minent_step(m, opt, images, labels, images_t)
        elif name == "advent":
            def fn(images, labels, images_t, m=m, d=d, opt=opt, opt_d=opt_d):
                return T.train_advent_step(m, d, opt, opt_d, images, labels, images_t)
        else:
            def fn(images, labels, images_t, m=m, d=d, opt=opt, opt_d=opt_d):
                return T.train_da_step(m, d, opt, opt_d, images, labels, images_t)
        graphs[name] = T.GraphedStep(fn, dict(images=x, labels=labels, images_t=xt), warmup=3,
                                     optimizers=[opt] if name == "minent" else [opt, opt_d])
    for gs in graphs.values():
        for _ in range(args.replays):
            gs()
    torch.cuda.synchronize()
    ms = {k: [] for k in graphs}
    for _ in range(args.repeats):
        for k, gs in graphs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.replays):
                gs.graph.replay()
            e1.record()
            torch.cuda.synchronize()
            ms[k].append(e0.elapsed_time(e1) / args.replays)
    out = {k: spread(v) for k, v in ms.items()}
    out["losses_last_replay"] = {k: [float(v) for v in gs.outputs] for k, gs in graphs.items()}
    out["advent_minus_da_step_ms"] = round(out["advent"]["median"] - out["da_step"]["median"], 4)
    return out


def bench_kernels(args):
    g = torch.Generator().manual_seed(1)
    h, w = H // 8, W // 8
    lr = (3 * torch.randn(N, h, w, 32, generator=g)).cuda()
    labels = torch.randint(0, NCLS, (N, H, W), generator=g).cuda()
    d_lr = torch.zeros_like(lr)
    acc = torch.zeros(2, dtype=torch.float64, device="cuda")
    bordered = torch.empty((N, H + 2, W + 2, 32), dtype=torch.bfloat16, device="cuda")
    bordered2 = torch.empty_like(bordered)
    K.upsample_fwd(lr, H, W, NCLS, K.UP_SOFTMAX, out=bordered2, out_flag=2, p_ld=32)
    K.entropy_fwd(lr, H, W, NCLS, K.ENT_MAP, emap=bordered, layout=K.MAP_ZERO_BORDERED)
    dmap = (torch.randn(bordered.shape, generator=g) * 1e-3).to(torch.bfloat16).cuda()
    calls = {
        "ce_training_pass": lambda: K.upsample_bwd(lr, H, W, NCLS, K.UP_CE, d_lr, labels=labels, loss_acc=acc),
        "entropy_training_pass": lambda: K.entropy_bwd(lr, H, W, NCLS, K.ENT_TRAIN, d_lr, acc=acc),
        "softmax_fwd": lambda: K.upsample_fwd(lr, H, W, NCLS, K.UP_SOFTMAX, out=bordered2, out_flag=2, p_ld=32),
        "self_info_fwd": lambda: K.entropy_fwd(lr, H, W, NCLS, K.ENT_MAP, emap=bordered, layout=K.MAP_ZERO_BORDERED),
        "softmax_bwd": lambda: K.upsample_bwd(lr, H, W, NCLS, K.UP_SOFTMAX, d_lr, grad_in=dmap, grad_is_bf16=2, p_ld=32),
        "self_info_bwd": lambda: K.entropy_bwd(lr, H, W, NCLS, K.ENT_SELF_INFO, d_lr, d_map=dmap,
                                               layout=K.MAP_ZERO_BORDERED),
        "entropy_fwd_sum_only": lambda: K.entropy_fwd(lr, H, W, NCLS, K.ENT_SUM, acc=acc),
    }
    launches = 50
    for fn in calls.values():
        for _ in range(5):
            fn()
    torch.cuda.synchronize()
    us = {k: [] for k in calls}
    for _ in range(args.repeats):
        for k, fn in calls.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(launches):
                fn()
            e1.record()
            torch.cuda.synchronize()
            us[k].append(1e3 * e0.elapsed_time(e1) / launches)
    out = {k: spread(v) for k, v in us.items()}
    med = {k: v["median"] for k, v in out.items()}
    lr_bytes = N * h * w * 32 * 4
    map_bytes = N * H * W * 32 * 2
    gbs = lambda nbytes, u: round(nbytes / (u * 1e-6) / 1e9, 1)  # noqa: E731
    out["ratios"] = {
        "entropy_training_pass / ce_training_pass": round(med["entropy_training_pass"] / med["ce_training_pass"], 3),
        "self_info_fwd / softmax_fwd": round(med["self_info_fwd"] / med["softmax_fwd"], 3),
        "self_info_bwd / softmax_bwd": round(med["self_info_bwd"] / med["softmax_bwd"], 3),
    }
    out["targets"] = {"entropy_training_pass / ce_training_pass": 1.25, "self_info_fwd / softmax_fwd": 1.15,
                      "self_info_bwd / softmax_bwd": 1.25}
    out["gbs_algorithmic"] = {
        "self_info_fwd": gbs(lr_bytes + map_bytes, med["self_info_fwd"]),
        "softmax_fwd": gbs(lr_bytes + map_bytes, med["softmax_fwd"]),
        "self_info_bwd": gbs(3 * lr_bytes + map_bytes, med["self_info_bwd"]),
        "softmax_bwd": gbs(3 * lr_bytes + map_bytes, med["softmax_bwd"]),
        "bytes_note": "fwd: logits fp32 32 floats/px once + bf16 map 64 B/px; bwd: + d_lr read and written",
    }
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--replays", type=int, default=20)
    ap.add_argument("--out", default=None, help="write the JSON result here (default: stdout only)")
    args = ap.parse_args()
    torch.backends.cudnn.allow_tf32 = False
    result = {"card": card(), "shape": "%d + %d images of %dx%d, %d classes, FCDiscriminator" % (N, N, H, W, NCLS)}
    result["kernels_us"] = bench_kernels(args)
    result["steps_ms"] = bench_steps(args)
    result["step_target"] = "advent <= da_step + 0.3 ms"
    text = json.dumps(result, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
