"""Generates the golden vectors that pin ``oracle/`` to the UNMODIFIED reference.

Run in the build container only (``/root/reference`` does not exist on the GPU box):

    PYTHONDONTWRITEBYTECODE=1 python tests/golden/make_golden.py

It imports the reference's own ``model.*`` / ``utils`` modules, loads the deterministic synthetic
weights of ``oracle.segnet_oracle.make_*_state`` into them, runs them on seeded inputs (fp32, CPU)
and stores strided samples + checksums of the results in ``tests/golden/*.npz|json``.
"""
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = "/root/reference"
sys.path.insert(0, ROOT)
sys.path.insert(0, REF)
sys.dont_write_bytecode = True

from oracle import segnet_oracle as O  # noqa: E402

from model.model_stages import BiSeNet  # noqa: E402  (reference)
from model.discriminator import (FCDiscriminator, DepthWiseSepFCDiscriminator,  # noqa: E402
                                 DepthWiseSepBNFCDiscriminator)
import utils as ref_utils  # noqa: E402


def sample(t, step=97):
    a = t.detach().double().reshape(-1).numpy()
    return np.concatenate([a[::step], [a.sum(), np.abs(a).sum(), float(a.size)]])


def load_into(module, sd):
    own = module.state_dict()
    for k, v in sd.items():
        assert k in own and own[k].shape == v.shape, k
        own[k] = v.clone()
    module.load_state_dict(own)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(8)
    out = {}
    layout = {}

    # ---- key layouts -------------------------------------------------------------------------
    net = BiSeNet("STDCNet813", 19)
    layout["bisenet"] = [[k, list(v.shape), str(v.dtype)] for k, v in net.state_dict().items()]
    layout["bisenet_param_names"] = [n for n, _ in net.named_parameters()]
    for name, cls in (("dense", FCDiscriminator), ("dwsep", DepthWiseSepFCDiscriminator),
                      ("dwsep_bn", DepthWiseSepBNFCDiscriminator)):
        layout["disc_" + name] = [[k, list(v.shape), str(v.dtype)] for k, v in cls(19).state_dict().items()]
    shipped = torch.load(os.path.join(REF, "GTA5_model/GTA5_10_D1.pth"), map_location="cpu")
    layout["shipped_D1"] = [[k, list(v.shape), str(v.dtype)] for k, v in shipped.items()]
    with open(os.path.join(HERE, "state_dict_layout.json"), "w") as f:
        json.dump(layout, f)

    # ---- segmentation net --------------------------------------------------------------------
    sd = O.make_bisenet_state(seed=11, randomize_bn=True)
    load_into(net, sd)
    g = torch.Generator().manual_seed(5)
    x = torch.randn(2, 3, 64, 128, generator=g)
    labels = torch.randint(0, 20, (2, 64, 128), generator=g)
    labels[labels == 19] = 255
    net.eval()
    with torch.no_grad():
        o, o16, o32 = net(x)
    out["eval_out"], out["eval_out16"], out["eval_out32"] = sample(o), sample(o16), sample(o32)
    # eval metric path (train.py:36-47), one image at a time
    hist = np.zeros((19, 19))
    for i in range(2):
        pred = ref_utils.reverse_one_hot(o[i]).numpy()
        hist += ref_utils.fast_hist(labels[i].numpy().flatten(), pred.flatten(), 19)
    out["eval_hist"] = hist
    out["eval_iu"] = ref_utils.per_class_iu(hist)

    net.train()
    o, o16, o32 = net(x)
    ce = torch.nn.CrossEntropyLoss(ignore_index=255)
    loss = ce(o, labels) + ce(o16, labels) + ce(o32, labels)
    loss.backward()
    out["train_out"] = sample(o)
    out["train_loss"] = np.array([loss.item()])
    grads = {n: p.grad for n, p in net.named_parameters() if p.grad is not None}
    out["train_grad_names"] = np.array(sorted(grads.keys()))
    for n in ("cp.backbone.features.0.conv.weight", "cp.backbone.features.5.conv_list.2.conv.weight",
              "cp.arm32.conv_atten.weight", "ffm.conv1.weight", "conv_out.conv_out.weight",
              "cp.backbone.features.4.avd_layer.0.weight", "cp.conv_avg.bn.weight"):
        out["grad:" + n] = sample(grads[n], 13)
    out["train_running_mean"] = sample(net.state_dict()["cp.backbone.features.3.conv_list.1.bn.running_mean"], 1)

    # ---- OHEM (utils.py:256-271) -------------------------------------------------------------
    lab2 = torch.randint(0, 19, (2, 64, 128), generator=g)
    with torch.no_grad():
        for thr, keep in ((0.3567, 1024), (5.0, 1024), (0.3567, 16000)):
            v = ref_utils.OHEM_CrossEntroy_Loss(thr, keep)(o.detach(), lab2)
            out["ohem_%g_%d" % (thr, keep)] = np.array([v.item()])
    out["ohem_labels"] = lab2.numpy().astype(np.int16)

    # ---- discriminators ----------------------------------------------------------------------
    p = torch.softmax(torch.randn(2, 19, 64, 128, generator=g), dim=1)
    for name, cls in (("dense", FCDiscriminator), ("dwsep", DepthWiseSepFCDiscriminator),
                      ("dwsep_bn", DepthWiseSepBNFCDiscriminator)):
        d = cls(19)
        load_into(d, O.make_discriminator_state(name, seed=3))
        d.train()
        pin = p.clone().requires_grad_(True)
        y = d(pin)
        l = torch.nn.BCEWithLogitsLoss()(y, torch.zeros_like(y))
        l.backward()
        out["disc_%s_out" % name] = sample(y, 1)
        out["disc_%s_loss" % name] = np.array([l.item()])
        out["disc_%s_dinput" % name] = sample(pin.grad, 211)
        out["disc_%s_dclassifier" % name] = sample(d.classifier.weight.grad, 17)

    # ---- fast_hist / per_class_iu known answers (utils.py:161-172) -----------------------------
    rng = np.random.default_rng(7)
    a = rng.integers(-2, 22, size=5000).astype(np.int64)
    a[::50] = 255
    b = rng.integers(0, 19, size=5000).astype(np.int64)
    out["kat_a"], out["kat_b"] = a.astype(np.int16), b.astype(np.int16)
    h = ref_utils.fast_hist(a, b, 19)
    out["kat_hist"] = h
    out["kat_iu"] = ref_utils.per_class_iu(h)
    out["kat_iu_empty"] = ref_utils.per_class_iu(np.zeros((19, 19)))
    out["kat_iu_perfect"] = ref_utils.per_class_iu(np.diag(np.arange(1, 20)))
    out["x"] = x.numpy()
    out["labels"] = labels.numpy().astype(np.int16)
    out["disc_in_sample"] = sample(p)   # the test regenerates the input from seed 5 (keeps the file under 1 MB)
    np.savez_compressed(os.path.join(HERE, "reference_vectors.npz"), **out)
    print("wrote", len(out), "arrays")


if __name__ == "__main__":
    main()
