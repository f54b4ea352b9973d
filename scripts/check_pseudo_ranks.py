"""pseudo_label_thresholds over two NCCL ranks with different shards equals the single-process result over
the concatenated shards, bit for bit, on both ranks.

    python -m torch.distributed.run --nproc-per-node 2 scripts/check_pseudo_ranks.py

Each rank builds both shards from the same seeds (rank 0: 3 batches, rank 1: 2 batches of other sizes), runs
the selection over its own shard under NCCL, and compares with its own single-process run over all five
batches.  Exits non-zero on any difference."""
import os
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from dasemanticsegmentationaml_b200 import train as T  # noqa: E402


def shards(n):
    g = torch.Generator().manual_seed(11)
    sizes = [[(4, 256, 512), (2, 255, 511), (1, 97, 301)], [(3, 256, 512), (5, 64, 128)]]
    out = []
    for shard in sizes:
        preds, confs = [], []
        for shape in shard:
            preds.append(torch.randint(0, n, shape, generator=g).to(torch.uint8).cuda())
            confs.append((1 - 0.1 * torch.rand(shape, generator=g) ** 3).cuda())
        out.append((preds, confs))
    return out


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl")
    from dasemanticsegmentationaml_b200 import _lib
    _lib.set_device_index(local)
    ok = True
    for n, portion, cap in ((19, 0.5, 0.9), (32, 0.2, 1.0)):
        parts = shards(n)
        thr, counts = T.pseudo_label_thresholds(*parts[rank], n, portion, cap)
        # the single-process result over the union: computed with the world treated as one process
        all_p = parts[0][0] + parts[1][0]
        all_c = parts[0][1] + parts[1][1]
        world = T._world
        T._world = lambda: 1
        try:
            rthr, rcounts = T.pseudo_label_thresholds(all_p, all_c, n, portion, cap)
        finally:
            T._world = world
        same = torch.equal(counts, rcounts) and torch.equal(thr.view(torch.int32), rthr.view(torch.int32))
        print("rank %d n=%d portion=%g: counts %d pixels, thresholds %s the single-process result"
              % (rank, n, portion, int(counts.sum()), "equal" if same else "DIFFER from"), flush=True)
        ok &= same
    dist.destroy_process_group()
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
