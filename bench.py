#!/usr/bin/env python
"""Benchmark of the north-star hot path: the adversarial domain-adaptation train step
(BiSeNet-STDC813 + discriminator, forward/backward/update) on synthetic Cityscapes/GTAV-shaped data.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path, one rank per GPU
    python bench.py --impl reference --steps K --warmup W    # the reference algorithm on the host CPU
    python bench.py --workload eval --gpus 8                 # BASELINE config 5: sharded 1024x2048 eval

Prints ONE JSON line (rank 0).  `value` is whole-job source images per second with the inputs
resident in HBM; `e2e` is the same step driven from pinned HOST buffers through the public API
(H2D copies and the D2H read of the losses inside the timed region).  See DESIGN.md "Measurement".
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

H, W, BATCH, NCLS = 512, 1024, 8, 19
WORKLOADS = {
    "da_dense": "config[2]: adversarial DA train step, FCDiscriminator, 512x1024, batch 8/GPU",
    "da_dwsep": "config[3]: DA train step, DepthWiseSepFCDiscriminator, 512x1024, batch 8/GPU",
    "da_dwsep_bn": "config[3]: DA train step, DepthWiseSepBNFCDiscriminator, 512x1024, batch 8/GPU",
    "supervised": "config[1]: supervised train step (3x CE), 720x1280, batch 8",
    "supervised_ohem": "config[1]: supervised train step (3x OHEM CE, radix select), 720x1280, batch 8",
    "eval": "config[4]: full-resolution eval (train.val: forward + fused argmax + 19x19 confusion matrix, "
            "images sharded over the ranks, NCCL int64 sum), 1024x2048",
}
# algorithmic dense-conv FLOPs per (source, target) pair / image (BASELINE.md section 3)
GFLOP_PER_UNIT = {"da_dense": 444.87, "da_dwsep": 226.0, "da_dwsep_bn": 226.0, "supervised": 186.14,
                  "supervised_ohem": 186.14, "eval": 141.04}
SHAPES = {"supervised": (720, 1280), "supervised_ohem": (720, 1280), "eval": (1024, 2048)}
# entry points whose launches are tensor-core GEMMs (everything else with a byte count is HBM-bound)
GEMM_ENTRIES = ("b200_conv_igemm", "b200_conv_wgrad")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=None)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="da_dense", choices=sorted(WORKLOADS))
    ap.add_argument("--torch-optim", action="store_true", help="torch's fused SGD/Adam instead of optim.FusedSGD/FusedAdam")
    ap.add_argument("--batch", type=int, default=BATCH)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-profile", action="store_true")
    ap.add_argument("--profile-ahead-ms", type=float, default=60.0,
                    help="park the stream behind a spin kernel of this length before the profiled eager step, so the "
                         "per-launch CUDA events bracket device time, not the host's launch latency (0 = off)")
    ap.add_argument("--no-extras", action="store_true", help="skip the short runs of the other BASELINE configs")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of one CUDA graph per step")
    ap.add_argument("--profile-json", default=None, help="write the per-kernel time table here")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (returned values; for a train step also "
                         "the parameters and BatchNorm statistics it left) as DIR/<name>.npy, for comparing two builds")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    return args


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sustained=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    source="MEASURED_PEAKS.json")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sustained=1400.0, source="fallback (B200_PROFILING.md)")


# --------------------------------------------------------------------------- CPU reference arm
def cpu_da_step_rate(workload, batch, steps, warmup, threads=None):
    """Oracle port of the reference step (fp32, CPU, all host threads): images per second."""
    import torch
    from oracle import segnet_oracle as O
    # every host core this process may use (torchrun exports OMP_NUM_THREADS=1: override it)
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    torch.set_num_threads(threads or avail)
    kind = {"da_dense": "dense", "da_dwsep": "dwsep", "da_dwsep_bn": "dwsep_bn"}.get(workload)
    h, w = SHAPES.get(workload, (H, W))
    g = torch.Generator().manual_seed(0)
    seg = O.clone_state(O.make_bisenet_state(seed=0), requires_grad=True)
    opt = torch.optim.SGD([v for v in seg.values() if v.requires_grad], lr=0.01, momentum=0.9, weight_decay=5e-4)
    x = torch.randn(batch, 3, h, w, generator=g)
    xt = torch.randn(batch, 3, h, w, generator=g)
    labels = torch.randint(0, NCLS, (batch, h, w), generator=g)
    if kind:
        dsd = O.clone_state(O.make_discriminator_state(kind, seed=1), requires_grad=True)
        opt_d = torch.optim.Adam([v for v in dsd.values() if v.requires_grad], lr=1e-3, betas=(0.9, 0.99))

    def step():
        if workload == "eval":
            with torch.no_grad():
                O.eval_batch(seg, x, labels)
        elif kind:
            O.da_step(seg, dsd, kind, x, labels, xt, opt, opt_d)
        else:
            opt.zero_grad()
            loss, _ = O.supervised_loss(seg, x, labels, True)
            loss.backward()
            opt.step()

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = time.perf_counter() - t0
    return batch * steps / dt, dt / steps * 1e3, torch.get_num_threads()


def _cpu_batch(workload, want):
    """Largest batch <= want whose fp32 autograd step fits the host's free memory (about 5 GB per
    512x1024 image pair, activations + gradients of the fp32 oracle)."""
    try:
        import psutil
        free = psutil.virtual_memory().available / 2 ** 30
    except Exception:
        free = 32.0
    h, w = SHAPES.get(workload, (H, W))
    per_img = 5.0 * (h * w) / (H * W)
    b = want
    while b > 2 and b * per_img > 0.7 * free:
        b //= 2
    return b


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps = args.steps or 2
    warmup = args.warmup if args.warmup is not None else 1
    # the SAME configuration as the GPU arm (batch 8 per step) whenever the host memory allows it;
    # BatchNorm on the 1x1 pooled maps needs >= 2 images per step in any case
    batch = _cpu_batch(args.workload, args.batch)
    rate, ms, threads = cpu_da_step_rate(args.workload, batch, steps, warmup)
    h, w = SHAPES.get(args.workload, (H, W))
    sample = ("%d-image %s step(s) of the oracle port (fp32, torch CPU), %d warm-up%s"
              % (batch, args.workload, warmup,
                 "" if batch == args.batch else "; a bounded sample of the %d-image step of `config` (the host's free memory / the "
                 "time limit): the per-image rate of the port grows a few per cent with the batch" % args.batch))
    line = {
        "impl": "reference", "metric": _metric(args.workload),
        "value": rate, "unit": "img/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        # the GPU arm's workload; `sample_batch` is what one timed CPU step actually processed
        "config": {"workload": WORKLOADS[args.workload], "batch_per_gpu": args.batch, "height": h, "width": w, "classes": NCLS,
                   "sample_batch": batch},
        "cpu_baseline": {"value": rate, "unit": "img/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def _metric(workload):
    if workload.startswith("da_"):
        return "da_train_step_img_per_s"
    return "eval_img_per_s" if workload == "eval" else "train_step_img_per_s"


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons, sampled every 100 ms from before the warm-up; stop()
    summarises the samples whose timestamps fall inside the timed window."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self, t0, t1):
        import datetime
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        rows = []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in out.strip().splitlines():
            f = [t.strip() for t in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), float(f[3]),
                             [n for n, v in zip(names, f[4:8]) if v.lower().startswith("active")]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 - 0.05 <= r[0] <= t1 + 0.05]
        window = "timed region"
        if not inside and rows:  # region shorter than the sampling period: take the closest samples
            inside = sorted(rows, key=lambda r: abs(r[0] - 0.5 * (t0 + t1)))[:3]
            window = "nearest samples (timed region shorter than the 100 ms period)"
        sm = sorted(r[1] for r in inside)
        reasons = sorted(set(n for r in inside for n in r[4]))
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max([r[2] for r in inside]) if inside else None,
                "power_w_max": max([r[3] for r in inside]) if inside else None, "samples": len(inside),
                "window": window, "reasons": reasons}


# --------------------------------------------------------------------------- B200 arm
class Bench(object):
    """One workload on this rank's GPU: models, optimizers, synthetic host + device buffers."""

    def __init__(self, args, workload, rank, world, dev, batch):
        import torch
        from dasemanticsegmentationaml_b200 import optim as B200Optim
        from dasemanticsegmentationaml_b200.model import (BiSeNet, FCDiscriminator, DepthWiseSepFCDiscriminator,
                                                          DepthWiseSepBNFCDiscriminator)
        self.args, self.workload, self.rank, self.world, self.dev, self.nb = args, workload, rank, world, dev, batch
        self.h, self.w = SHAPES.get(workload, (H, W))
        torch.manual_seed(0)  # identical initial weights on every rank
        self.model = BiSeNet("STDCNet813", NCLS).to(dev)
        # same optimizers and hyper-parameters as train.py:170-172
        if args.torch_optim:
            self.opt = torch.optim.SGD(self.model.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4, fused=True)
        else:   # one launch per optimizer step (SURVEY 8 f3); same arithmetic as torch.optim.SGD / Adam
            self.opt = B200Optim.FusedSGD(self.model.parameters(), lr=0.01, momentum=0.9, weight_decay=5e-4)
        self.model_d = self.opt_d = None
        if workload.startswith("da_"):
            cls = {"da_dense": FCDiscriminator, "da_dwsep": DepthWiseSepFCDiscriminator,
                   "da_dwsep_bn": DepthWiseSepBNFCDiscriminator}[workload]
            self.model_d = cls(NCLS).to(dev)
            if args.torch_optim:
                self.opt_d = torch.optim.Adam(self.model_d.parameters(), lr=1e-3, betas=(0.9, 0.99), fused=True, capturable=True)
            else:
                self.opt_d = B200Optim.FusedAdam(self.model_d.parameters(), lr=1e-3, betas=(0.9, 0.99))
        # the seeded start that restore() returns to before every timed step
        self.state = [t.detach() for m in (self.model, self.model_d) if m is not None
                      for t in list(m.parameters()) + list(m.buffers())]
        self.state0 = [t.clone() for t in self.state]
        self.host = self.make_host(rank)
        self.devbuf = {k: v.to(dev) for k, v in self.host.items()}
        self.names = [k for k in self.devbuf if not (self.model_d is None and k == "images_t")]
        self.graphed = None
        self.graph_note = "eager (--no-graph)"
        self.eval_state = {}

    def make_host(self, rank, pin=True):
        import torch
        g = torch.Generator().manual_seed(100 + rank)  # rank-dependent data
        host = {
            "images": torch.randn(self.nb, 3, self.h, self.w, generator=g),
            "labels": torch.randint(0, NCLS + 1, (self.nb, self.h, self.w), generator=g),
            "images_t": torch.randn(self.nb, 3, self.h, self.w, generator=g),
        }
        if self.workload == "supervised_ohem":
            host["labels"].clamp_(max=NCLS - 1)  # the reference's OHEM has no ignore_index
        else:
            host["labels"][host["labels"] == NCLS] = 255
        if self.workload == "eval":
            del host["images_t"]
        return {k: (v.pin_memory() if pin else v) for k, v in host.items()}

    def restore(self):
        """Puts the models and optimizers back to their seeded start, in place (a captured graph reads
        these tensors): parameters and buffers as initialised, optimizer state zeroed, which is where a
        fresh SGD / Adam starts (no momentum, no moments, step count 0).  The adversarial training
        amplifies the last-bit differences of the fp32 atomic reductions from step to step, so steps
        that build on each other compute something different on every run; steps that all start here
        compute the same up to rounding."""
        import torch
        with torch.no_grad():
            torch._foreach_copy_(self.state, self.state0)
            opt_state = [t for o in (self.opt, self.opt_d) if o is not None
                         for st in o.state.values() for t in st.values() if torch.is_tensor(t)]
            if opt_state:
                torch._foreach_zero_(opt_state)

    def eager_step(self, buf):
        from dasemanticsegmentationaml_b200 import train as T
        if self.workload == "eval":
            # the reference's val() (train.py:24-61) over this rank's shard: forward, argmax, confusion
            # matrix on the device, ONE all-reduce + ONE device->host copy per evaluation
            import torch
            precision, miou = T.val(self.model, [(buf["images"], buf["labels"])], NCLS)
            self.eval_state = {"precision": precision, "miou": miou, "hist": T.val.last_hist}
            return (torch.tensor(miou, device=self.dev),)
        if self.workload == "supervised_ohem":
            return (T.train_step(self.model, self.opt, buf["images"], buf["labels"], loss="ohem"),)
        if self.model_d is None:
            return (T.train_step(self.model, self.opt, buf["images"], buf["labels"]),)
        return T.train_da_step(self.model, self.model_d, self.opt, self.opt_d, buf["images"], buf["labels"], buf["images_t"])

    def capture(self):
        from dasemanticsegmentationaml_b200 import train as T
        import torch
        if self.args.no_graph or self.workload == "eval":   # val() ends in a host read: nothing to replay
            if self.workload == "eval":
                self.graph_note = "eager (train.val ends with a device->host copy of the confusion matrix)"
            return
        try:
            self.graphed = T.GraphedStep(lambda **kw: self.eager_step(dict(self.devbuf, **kw)),
                                         {k: self.devbuf[k] for k in self.names},
                                         optimizers=[o for o in (self.opt, self.opt_d) if o is not None and not self.args.torch_optim])
            self.graph_note = "whole step replayed as one CUDA graph"
        except Exception as ex:  # capture is an optimisation: report and fall back to eager launches
            self.graphed = None
            self.graph_note = "eager (graph capture failed: %r)" % (ex,)
            torch.cuda.synchronize()

    def step(self, buf):
        if self.graphed is None:
            return self.eager_step(buf)
        if buf is self.devbuf:  # already in the graph's static buffers
            return self.graphed()
        return self.graphed(**{k: buf[k] for k in self.names})


def sync_all(world):
    import torch
    import torch.distributed as dist
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def time_resident(b, steps, warmup, clocks=None, dump_dir=None):
    """Timed region 1: inputs resident in HBM.  -> (ms per step (max over ranks), launches, losses, clk, host ms)
    Every step starts from the seeded state (Bench.restore, queued between the steps and outside their
    event pairs), so with the same arguments each step computes the same every run.
    dump_dir: rank 0 writes the last timed step's outputs there (dump_outputs)."""
    import torch
    import torch.distributed as dist
    from dasemanticsegmentationaml_b200 import _lib
    for _ in range(warmup):
        b.restore()
        b.step(b.devbuf)
    sync_all(b.world)
    t_wall0 = time.time()
    l0 = _lib.launch_count
    events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    host_s = 0.0
    for e0, e1 in events:
        b.restore()
        e0.record()
        t_host0 = time.perf_counter()
        losses = b.step(b.devbuf)
        host_s += time.perf_counter() - t_host0
        e1.record()
    host_enqueue_ms = host_s * 1e3 / steps  # host time to queue one step
    sync_all(b.world)
    t_wall1 = time.time()
    if dump_dir and b.rank == 0:   # before the launch count below, whose eager step moves the weights again
        dump_outputs(b, losses, dump_dir)
    launches = _lib.launch_count - l0
    if b.graphed is not None:  # replays do not pass through the binding: count one eager step's launches
        l1 = _lib.launch_count
        b.eager_step(b.devbuf)
        torch.cuda.synchronize()
        launches = (_lib.launch_count - l1) * steps
    ms = torch.tensor([sum(e0.elapsed_time(e1) for e0, e1 in events)], device=b.dev)
    if b.world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    clk = clocks.stop(t_wall0, t_wall1) if clocks else None
    return float(ms.item()) / steps, launches, [float(v) for v in losses], clk, host_enqueue_ms


def time_e2e(b, steps):
    """Timed region 2: end to end from pinned host buffers.  Every step copies ITS inputs
    host->device (pinned memory, a dedicated copy stream, double buffered so that the copy of step
    i+1 overlaps the compute of step i) and reads the step's result back to the host (one D2H +
    sync per step, as train.py's .item() calls do).  -> (ms per step, h2d bytes, d2h bytes)"""
    import torch
    import torch.distributed as dist
    names = b.names
    stage = [{k: torch.empty_like(b.devbuf[k]) for k in names} for _ in range(2)]
    for sbuf in stage:
        if "images_t" not in sbuf and "images_t" in b.devbuf:
            sbuf["images_t"] = b.devbuf["images_t"]
    h2d = sum(b.host[k].numel() * b.host[k].element_size() for k in names)
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]

    def issue_copy(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])      # the step that last used this slot is done
            for k in names:
                stage[slot][k].copy_(b.host[k], non_blocking=True)
            ready[slot].record(copy_stream)

    sync_all(b.world)
    for ev in consumed:
        ev.record()
    d2h_stream = torch.cuda.Stream()
    host_buf = torch.empty(8, dtype=torch.float32).pin_memory()

    def read_back(item):
        """Blocking D2H read of one step's stacked results on a side stream (waits for THAT step only)."""
        stacked, done = item
        with torch.cuda.stream(d2h_stream):
            d2h_stream.wait_event(done)
            host_buf[:stacked.numel()].copy_(stacked, non_blocking=True)
        d2h_stream.synchronize()
        return host_buf[:stacked.numel()].clone()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    issue_copy(0)
    pending = None
    n_out = 1
    for i in range(steps):
        slot = i & 1
        if i + 1 < steps:
            issue_copy(slot ^ 1)
        torch.cuda.current_stream().wait_event(ready[slot])
        out = b.step(stage[slot])
        consumed[slot].record()
        stacked = torch.stack([o.float() for o in out])
        n_out = len(out)
        done = torch.cuda.Event()
        done.record()
        # every step's results are read back to the host; the read of step i happens after step i+1
        # has been queued, so the host-side sync never leaves the GPU idle
        if pending is not None:
            read_back(pending)
        pending = (stacked, done)
    read_back(pending)
    e1.record()
    sync_all(b.world)
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=b.dev)
    if b.world > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    d2h = 4 * n_out + (8 * NCLS * NCLS if b.workload == "eval" else 0)   # eval: + the int64 confusion matrix
    return float(ms2.item()) / steps, h2d, d2h


def weights_checksum(modules, buffers=False):
    """Bit-level checksum (int64 wrap-around sum of the fp32 bit patterns) of all parameters, or of all
    buffers (BatchNorm running statistics)."""
    import torch
    tot = torch.zeros((), dtype=torch.int64, device=next(modules[0].parameters()).device)
    for m in modules:
        for t in (list(m.buffers()) if buffers else list(m.parameters())):
            if t.dtype == torch.float32:
                tot += t.detach().contiguous().view(torch.int32).to(torch.int64).sum()
            else:
                tot += t.detach().to(torch.int64).sum()
    return tot


DUMP_LIMIT_BYTES = 64 * 10 ** 6


def dump_outputs(b, result, out_dir):
    """Writes what the last timed step computed as out_dir/<name>.npy: the values the step returns to its
    caller (float32; the host-side evaluation numbers and confusion matrix as float64) and, for a train
    step, the parameters and floating-point buffers (BatchNorm running statistics) of every model it
    updated, each flattened to one float32 vector in parameters() / buffers() order.  Inputs and initial
    weights are seeded, so two builds run with the same arguments can be compared file by file."""
    import numpy as np
    import torch
    if b.workload == "eval":
        st = b.eval_state
        arrays = {"precision": np.array([st["precision"]]), "miou": np.array([st["miou"]]),
                  "hist": st["hist"].cpu().numpy().reshape(NCLS, NCLS).astype(np.float64)}
    else:
        names = ("loss_seg", "loss_adv_g", "loss_d_src", "loss_d_tgt") if b.model_d is not None else ("loss",)
        assert len(names) == len(result), (names, len(result))
        arrays = {n: v.detach().float().reshape(1).cpu().numpy() for n, v in zip(names, result)}
        for tag, m in (("seg", b.model), ("disc", b.model_d)):
            if m is None:
                continue
            arrays[tag + "_params"] = torch.cat([p.detach().float().reshape(-1) for p in m.parameters()]).cpu().numpy()
            bufs = [t.detach().float().reshape(-1) for t in m.buffers() if t.is_floating_point()]
            if bufs:
                arrays[tag + "_buffers"] = torch.cat(bufs).cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        raise SystemExit("bench.py: --dump-outputs would write %d bytes, more than %d" % (total, DUMP_LIMIT_BYTES))
    os.makedirs(out_dir, exist_ok=True)
    for n, a in arrays.items():
        np.save(os.path.join(out_dir, n + ".npy"), a)


def dp_check(b):
    """Data-parallel consistency: after the timed steps every rank must hold bit-identical weights
    (same initial weights + identical averaged gradients); checked on a bit-level checksum."""
    import torch
    import torch.distributed as dist
    mods = [m for m in (b.model, b.model_d) if m is not None]
    mine = torch.stack([weights_checksum(mods), weights_checksum(mods, buffers=True)])
    if b.world == 1:
        return {"ranks": 1, "identical_on_all_ranks": True, "checksum": int(mine[0].item())}
    parts = [torch.empty_like(mine) for _ in range(b.world)]
    dist.all_gather(parts, mine)
    vals = [int(p[0].item()) for p in parts]
    bufs = [int(p[1].item()) for p in parts]
    # PARAMETERS must be bit-identical (same start + identical averaged gradients).  The BatchNorm running
    # statistics are per-GPU by design -- every rank normalises with its own batch, as the replicas of the
    # reference's nn.DataParallel do (train.py:145-152), which keeps only device 0's -- and are reported apart.
    return {"ranks": b.world, "identical_on_all_ranks": all(v == vals[0] for v in vals), "checksum": vals[0],
            "batchnorm_running_stats_identical": all(v == bufs[0] for v in bufs)}


def eval_hist_check(b):
    """BASELINE config 5: the all-reduced confusion matrix of the sharded evaluation must equal, bit for
    bit, the matrix ONE process computes over all ranks' images (rank 0 regenerates the other ranks'
    shards from their seeds and evaluates them itself with the same weights)."""
    import torch
    from dasemanticsegmentationaml_b200 import train as T
    import torch.distributed as dist
    summed = b.eval_state.get("hist")
    if summed is None:
        return None
    # (1) the collective: the all-reduced matrix must equal, bit for bit, the sum of the ranks' own matrices
    local = T.val.last_local_hist
    parts = [local]
    if b.world > 1:
        parts = [torch.empty_like(local) for _ in range(b.world)]
        dist.all_gather(parts, local)
    if b.rank != 0:
        return None
    host_sum = sum(p.cpu().numpy().astype("int64") for p in parts)
    # (2) one process over all shards: rank 0 regenerates the other ranks' images from their seeds and evaluates
    # them itself.  The forward is not bit-reproducible (the global-average-pool sums of the attention modules
    # are fp32 atomics), and on a random-init net most arg-maxes are near ties, so this is reported as the
    # fraction of pixels that land in another cell, not asserted.
    single = None
    with torch.no_grad():
        for r in range(b.world):
            host = b.make_host(r, pin=False)
            single, _ = T.eval_batch(b.model, host["images"].to(b.dev), host["labels"].to(b.dev), NCLS, single)
    moved = int((summed.cpu() - single.cpu()).abs().sum().item()) // 2
    valid = int(summed.sum().item())
    return {"ranks": b.world, "images": b.nb * b.world, "pixels": int(b.nb * b.world * b.h * b.w),
            "summed_hist_equals_sum_of_rank_hists": bool((summed.cpu().numpy() == host_sum).all()),
            "summed_hist_equals_single_process": bool(torch.equal(summed.cpu(), single.cpu())),
            "pixels_in_another_cell_when_recomputed": moved, "hist_total": valid,
            "valid_pixels_expected": int(sum(int((b.make_host(r, pin=False)["labels"] != 255).sum()) for r in range(b.world))),
            "precision": b.eval_state["precision"], "miou": b.eval_state["miou"]}


def run_b200(args):
    import torch
    import torch.distributed as dist
    from dasemanticsegmentationaml_b200 import _lib, build

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the B200 path has no CPU fallback (use --impl reference)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    if rank == 0:
        build.build()
    if world > 1:
        dist.barrier()
    _lib.ensure_device(local)
    _lib.set_device_index(local)

    steps = args.steps or 20
    warmup = max(3, args.warmup if args.warmup is not None else 5)
    b = Bench(args, args.workload, rank, world, dev, args.batch)
    for _ in range(2):      # eager warm-up (also fills lazy state), then capture the whole step
        b.eager_step(b.devbuf)
    b.capture()
    clocks = ClockSampler(local) if rank == 0 else None
    ms_step, launches, loss_vals, clk, host_ms = time_resident(b, steps, warmup, clocks, args.dump_outputs)
    e2e_ms, h2d, d2h = time_e2e(b, steps)
    check = eval_hist_check(b) if args.workload == "eval" else dp_check(b)

    # ---- per-kernel profile of ONE step (CUDA events around every launch of ours) -----------------
    prof = None
    if not args.no_profile:
        sync_all(world)
        # every launch timed ALONE: the profiled step keeps the small layers' weight gradients on the main stream
        # (in the timed steps they run beside the data gradients on a side stream, ops.SIDE)
        from dasemanticsegmentationaml_b200 import ops as _ops
        side, _ops.WGRAD_SIDE_MAX_PIXELS = _ops.WGRAD_SIDE_MAX_PIXELS, 0
        _lib.profile_start(host_ahead_ms=args.profile_ahead_ms)
        b.eager_step(b.devbuf)
        prof = _lib.profile_stop()
        _ops.WGRAD_SIDE_MAX_PIXELS = side
        detail = _lib.last_profile_detail

    if world > 1:
        dist.barrier()
    if rank != 0:
        _finish(world)
        return

    peaks = measured_peaks()
    nb, h, w = b.nb, b.h, b.w
    unit_per_step = nb * world
    value = unit_per_step / (ms_step / 1e3)
    line = {
        "metric": _metric(args.workload),
        "value": value, "unit": "img/s", "n_gpus": world, "steps": steps, "warmup": warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOADS[args.workload], "batch_per_gpu": nb, "height": h, "width": w,
                   "classes": NCLS, "parallelism": "dp%d" % world,
                   "l2": "inputs (134 MB/step) and activations (>1 GB/step) exceed the 126 MB L2; no explicit flush",
                   "pairs_per_s": value if b.model_d is not None else None,
                   "losses_last_step": loss_vals, "host_enqueue_ms_per_step": host_ms,
                   "launch_mode": b.graph_note,
                   ("eval_check" if args.workload == "eval" else "dp_check"): check},
        "e2e": {"value": unit_per_step / (e2e_ms / 1e3), "unit": "img/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms},
        "gpu_launches": launches,
        "clocks": clk,
    }
    step_tf = GFLOP_PER_UNIT[args.workload] * nb / 1e3 / (ms_step / 1e3)  # TFLOP/s per GPU, whole step
    line["config"]["step_algorithmic_tflops_per_gpu"] = step_tf
    if prof:
        add_rooflines(line, prof, peaks, args)
        if args.profile_json:
            with open(args.profile_json, "w") as f:
                json.dump({"by_kernel": prof, "by_shape": detail}, f, indent=1)
    del b
    torch.cuda.empty_cache()

    # ---- the other BASELINE configs, short runs (driver-observed numbers for configs 1, 3, 4) -----
    if world == 1 and not args.no_extras and args.workload == "da_dense":
        extras = {}
        for wl in ("da_dwsep", "da_dwsep_bn", "supervised_ohem", "eval"):
            try:
                eb = Bench(args, wl, rank, world, dev, args.batch)
                for _ in range(2):
                    eb.eager_step(eb.devbuf)
                eb.capture()
                ms_e, _, lv, _, _ = time_resident(eb, 5, 3)
                ent = {"workload": WORKLOADS[wl], "img_per_s": eb.nb / (ms_e / 1e3), "ms_per_step": ms_e, "steps": 5,
                       "warmup": 3, "height": eb.h, "width": eb.w, "launch_mode": eb.graph_note, "result_last_step": lv}
                if wl.startswith("da_dwsep"):
                    # BASELINE config 4 is judged by HBM GB/s: the depthwise / BatchNorm kernels of this step
                    from dasemanticsegmentationaml_b200 import ops as _ops
                    side, _ops.WGRAD_SIDE_MAX_PIXELS = _ops.WGRAD_SIDE_MAX_PIXELS, 0
                    _lib.profile_start(host_ahead_ms=args.profile_ahead_ms)
                    eb.eager_step(eb.devbuf)
                    pe = _lib.profile_stop()
                    _ops.WGRAD_SIDE_MAX_PIXELS = side
                    ent["roofline_mem"] = mem_table(pe, peaks, only=("b200_dwconv", "b200_bn_", "b200_upsample", "b200_act_bwd"))
                if wl == "eval":
                    ent["eval_check"] = eval_hist_check(eb)
                extras[wl] = ent
                del eb
            except Exception as ex:   # never lose the headline over an extra
                extras[wl] = {"failed": repr(ex)}
            torch.cuda.empty_cache()
        line["extra"] = extras

    if not args.no_cpu_baseline and world == 1 and args.workload != "supervised_ohem":
        try:
            cb_batch, cb_steps = min(4, args.batch), (4 if args.workload != "eval" else 2)
            rate, cms, threads = cpu_da_step_rate(args.workload, cb_batch, cb_steps, 1)
            line["cpu_baseline"] = {"value": rate, "unit": "img/s", "cores": threads, "kind": "port",
                                    "sample": "%d steps of %d source + %d target images (same %dx%d workload, reduced batch) "
                                              "of the oracle port, fp32 torch CPU, after one warm-up step; %.1f s per step"
                                              % (cb_steps, cb_batch, cb_batch, h, w, cms / 1e3)}
        except Exception as ex:  # the baseline is informational; never lose the GPU line over it
            line["cpu_baseline"] = {"value": None, "unit": "img/s", "cores": os.cpu_count(), "kind": "port",
                                    "sample": "failed: %r" % (ex,)}
    emit(line)
    _finish(world)


def mem_table(prof, peaks, only=None):
    """{entry point: achieved GB/s on its algorithmic bytes, fraction of the measured HBM copy rate}
    for the HBM-bound kernels of one eager step (CUDA events around each launch)."""
    out = {}
    for k, v in prof.items():
        if k in GEMM_ENTRIES or v["bytes"] <= 0 or v["ms"] <= 0:
            continue
        if only and not k.startswith(tuple(only)):
            continue
        gbs = v["bytes"] / (v["ms"] / 1e3) / 1e9
        out[k] = {"gbs": round(gbs, 1), "frac_of_hbm": round(gbs / peaks["hbm"], 3), "launches": v["calls"],
                  "ms": round(v["ms"], 3), "mbytes": round(v["bytes"] / 1e6, 1)}
    return out


def add_rooflines(line, prof, peaks, args):
    conv = prof.get("b200_conv_igemm")
    tot_ms = sum(v["ms"] for v in prof.values())
    table = sorted(((k, v["calls"], v["ms"], v["flops"]) for k, v in prof.items()), key=lambda r: -r[2])
    if conv and conv["ms"] > 0:
        ach = conv["flops"] / (conv["ms"] / 1e3) / 1e12
        traffic, traffic_src = conv_traffic(args.workload)
        line["roofline"] = {"bound": "tensor",
                            "kernel": "conv_igemm_pair_kernel (cta_group::2) + conv_igemm_kernel / conv_igemm_persistent_kernel "
                                      "(forward + data-gradient launches of b200_conv_igemm)",
                            "achieved": ach, "peak": peaks["tf_burst"], "unit": "TFLOP/s",
                            "frac": ach / peaks["tf_burst"], "traffic": traffic, "traffic_source": traffic_src,
                            "peak_source": peaks["source"] + " bf16_tflops (burst: every launch is timed alone with CUDA events)",
                            "frac_of_sustained": ach / peaks["tf_sustained"],
                            "launches_per_step": conv["calls"], "avg_launch_ms": conv["ms"] / conv["calls"],
                            "share_of_kernel_time": conv["ms"] / tot_ms}
    line["kernel_time_ms_per_step"] = {k: round(ms_, 3) for k, _, ms_, _ in table}
    wg = prof.get("b200_conv_wgrad")
    if wg and wg["ms"] > 0:
        line["wgrad_tflops"] = wg["flops"] / (wg["ms"] / 1e3) / 1e12
    line["roofline_mem"] = mem_table(prof, peaks)


def _finish(world):
    """Leave without tearing NCCL down: destroying a communicator that a live CUDA graph still
    references can block forever, and the process is exiting anyway."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        os._exit(0)


def conv_traffic(workload):
    """DRAM bytes per conv launch from the committed ncu capture (only measured for the default workload)."""
    for name in ("r2_conv_traffic.json", "r1_conv_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if workload == "da_dense" and os.path.exists(path):
            with open(path) as f:
                return json.load(f).get("traffic_bytes_per_launch"), \
                    "profiles/%s (ncu dram__bytes_read+write per launch, da_dense step)" % name
    return None, None


_REAL_FD = None


def emit(line):
    """The ONE JSON line of the contract goes to the real stdout; everything else any library or
    module prints while the bench runs (STDCNet813's 'use pretrain model' notice, kept for parity
    with stdcnet.py:139; NCCL's own "NCCL version ..." banner, written by the C library straight to
    file descriptor 1) is routed to stderr."""
    os.write(_REAL_FD, (json.dumps(line) + "\n").encode())


def main():
    global _REAL_FD
    args = parse()
    sys.stdout.flush()
    _REAL_FD = os.dup(1)      # keep the real stdout for the JSON line ...
    os.dup2(2, 1)             # ... and point fd 1 at stderr for everything else (C libraries included)
    sys.stdout = sys.stderr
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
