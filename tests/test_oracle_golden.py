"""Pins oracle/segnet_oracle.py to the unmodified reference through the committed golden vectors
(tests/golden/reference_vectors.npz, produced by tests/golden/make_golden.py from /root/reference)."""
import json
import os

import numpy as np
import pytest
import torch

from oracle import segnet_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def gold():
    return np.load(os.path.join(GOLD, "reference_vectors.npz"))


def sample(t, step=97):
    a = t.detach().double().reshape(-1).numpy()
    return np.concatenate([a[::step], [a.sum(), np.abs(a).sum(), float(a.size)]])


def close(a, b, rtol=2e-4, atol=2e-5):
    np.testing.assert_allclose(a, b, rtol=rtol, atol=atol)


def disc_input(gold):
    """The discriminator input of make_golden.py, regenerated from its seeded generator (the draw after
    x, labels and ohem_labels) instead of stored whole, and checked against the stored sample."""
    g = torch.Generator().manual_seed(5)
    torch.randn(2, 3, 64, 128, generator=g)
    torch.randint(0, 20, (2, 64, 128), generator=g)
    torch.randint(0, 19, (2, 64, 128), generator=g)
    p = torch.softmax(torch.randn(2, 19, 64, 128, generator=g), dim=1)
    close(sample(p), gold["disc_in_sample"], rtol=1e-6, atol=0)
    return p


def test_seg_eval_forward_and_metric(gold):
    torch.set_num_threads(8)
    sd = O.make_bisenet_state(seed=11, randomize_bn=True)
    x = torch.from_numpy(gold["x"])
    labels = torch.from_numpy(gold["labels"].astype(np.int64))
    outs = O.bisenet_forward(sd, x, training=False)
    close(sample(outs[0]), gold["eval_out"])
    close(sample(outs[1]), gold["eval_out16"])
    close(sample(outs[2]), gold["eval_out32"])
    _, hist = O.eval_batch(sd, x, labels)
    assert np.array_equal(hist, gold["eval_hist"].astype(np.int64))
    assert np.array_equal(O.per_class_iu(hist), gold["eval_iu"])


def test_seg_train_forward_backward(gold):
    torch.set_num_threads(8)
    sd = O.clone_state(O.make_bisenet_state(seed=11, randomize_bn=True), requires_grad=True)
    x = torch.from_numpy(gold["x"])
    labels = torch.from_numpy(gold["labels"].astype(np.int64))
    loss, outs = O.supervised_loss(sd, x, labels, training=True)
    loss.backward()
    close(sample(outs[0]), gold["train_out"])
    close(np.array([loss.item()]), gold["train_loss"], rtol=1e-5)
    with_grad = sorted(k for k, v in sd.items() if v.requires_grad and v.grad is not None)
    assert with_grad == list(gold["train_grad_names"])
    for key in gold.files:
        if key.startswith("grad:"):
            close(sample(sd[key[5:]].grad, 13), gold[key], rtol=2e-3, atol=1e-6)
    close(sample(sd["cp.backbone.features.3.conv_list.1.bn.running_mean"], 1), gold["train_running_mean"])


def test_ohem(gold):
    sd = O.make_bisenet_state(seed=11, randomize_bn=True)
    x = torch.from_numpy(gold["x"])
    with torch.no_grad():
        out = O.bisenet_forward(sd, x, training=True)[0]
    lab = torch.from_numpy(gold["ohem_labels"].astype(np.int64))
    for thr, keep in ((0.3567, 1024), (5.0, 1024), (0.3567, 16000)):
        v = O.ohem_cross_entropy(out, lab, thr, keep)
        close(np.array([v.item()]), gold["ohem_%g_%d" % (thr, keep)], rtol=1e-4)


@pytest.mark.parametrize("kind", ["dense", "dwsep", "dwsep_bn"])
def test_discriminators(gold, kind):
    sd = O.clone_state(O.make_discriminator_state(kind, seed=3), requires_grad=True)
    p = disc_input(gold).requires_grad_(True)
    y = O.discriminator_forward(kind, sd, p, training=True)
    loss = O.bce_with_logits_const(y, 0.0)
    loss.backward()
    close(sample(y, 1), gold["disc_%s_out" % kind])
    close(np.array([loss.item()]), gold["disc_%s_loss" % kind], rtol=1e-5)
    close(sample(p.grad, 211), gold["disc_%s_dinput" % kind], rtol=2e-3, atol=1e-9)
    close(sample(sd["classifier.weight"].grad, 17), gold["disc_%s_dclassifier" % kind], rtol=2e-3, atol=1e-8)


def test_fast_hist_known_answers(gold):
    a, b = gold["kat_a"].astype(np.int64), gold["kat_b"].astype(np.int64)
    h = O.fast_hist(a, b, 19)
    assert h.dtype == np.int64 and np.array_equal(h, gold["kat_hist"])
    assert np.array_equal(O.per_class_iu(h), gold["kat_iu"])
    assert np.array_equal(O.per_class_iu(np.zeros((19, 19))), gold["kat_iu_empty"])
    assert np.array_equal(O.per_class_iu(np.diag(np.arange(1, 20))), gold["kat_iu_perfect"])
    # edge cases probed on the reference: 255 / negative labels are dropped, empty input is all zeros
    assert O.fast_hist(np.array([255, -1, 19], dtype=np.int64), np.array([0, 1, 2], dtype=np.int64), 19).sum() == 0
    assert O.fast_hist(np.zeros(0, dtype=np.int64), np.zeros(0, dtype=np.int64), 19).shape == (19, 19)
    assert O.compute_global_accuracy(np.array([1, 2, 3]), np.array([1, 255, 3])) == pytest.approx(2 / 3)


def test_state_dict_layout_of_oracle_weights():
    layout = json.load(open(os.path.join(GOLD, "state_dict_layout.json")))
    ref = {k: tuple(s) for k, s, _ in layout["bisenet"]}
    sd = O.make_bisenet_state(seed=0)
    for k, v in sd.items():
        assert k in ref and tuple(v.shape) == ref[k], k
    for kind in ("dense", "dwsep", "dwsep_bn"):
        ref = [(k, tuple(s)) for k, s, _ in layout["disc_" + kind]]
        got = [(k, tuple(v.shape)) for k, v in O.make_discriminator_state(kind).items()]
        assert got == ref


@pytest.mark.parametrize("variant", ["da", "nni"])
def test_adversarial_step_loops(variant):
    """oracle.da_step / da_step_nni against the loop bodies of train.py:192-262 / train_nni.py:105-163
    replayed with the reference's own modules (tests/golden/make_golden_steps.py)."""
    torch.set_num_threads(8)
    gold = np.load(os.path.join(GOLD, "reference_steps.npz"))
    x, xt = torch.from_numpy(gold["x"]), torch.from_numpy(gold["xt"])
    labels = torch.from_numpy(gold["labels"].astype(np.int64)).squeeze(1)  # train.py:214 squeezes too
    sd = O.clone_state(O.make_bisenet_state(seed=31), requires_grad=True)
    dsd = O.clone_state(O.make_discriminator_state("dense", seed=6), requires_grad=True)
    opt = torch.optim.SGD([v for v in sd.values() if v.requires_grad], lr=0.01, momentum=0.9, weight_decay=5e-4)
    opt_d = torch.optim.Adam([v for v in dsd.values() if v.requires_grad], lr=1e-3, betas=(0.9, 0.99))
    step = O.da_step if variant == "da" else O.da_step_nni
    got = step(sd, dsd, "dense", x, labels, xt, opt, opt_d, lambda_adv=0.01)
    close(np.array(got), gold[variant + "_losses"], rtol=2e-4)
    for key in gold.files:
        if key.startswith(variant + ":"):
            close(sample(sd[key.split(":", 1)[1]], 7), gold[key], rtol=2e-3, atol=2e-6)
        if key.startswith(variant + "_d:"):
            close(sample(dsd[key.split(":", 1)[1]], 7), gold[key], rtol=2e-3, atol=2e-6)


@pytest.mark.parametrize("tag,block,last", [("add", "add", False), ("cat_last", "cat", True)])
def test_backbone_variants_against_reference(tag, block, last):
    """AddBottleneck (stdcnet.py:17-64) and use_conv_last (stdcnet.py:126,191-192) restatements vs
    golden vectors of the reference's own STDCNet813(type=..., use_conv_last=...)."""
    torch.set_num_threads(8)
    gold = np.load(os.path.join(GOLD, "reference_backbone.npz"))

    def smp(t, step=53):
        return sample(t, step)

    x = torch.from_numpy(gold["x"])
    sd = O.clone_state(O.make_backbone_state(seed=17, block=block, use_conv_last=last), requires_grad=True)
    feats = O.stdcnet813(sd, "bb", x, True, block=block, use_conv_last=last)
    gw = torch.Generator().manual_seed(22)
    loss = sum((f * torch.randn(f.shape, generator=gw)).sum() for f in feats)
    loss.backward()
    for i, f in enumerate(feats):
        close(smp(f), gold["%s_feat%d" % (tag, i)])
    n_grad = 0
    for key in gold.files:
        if key.startswith(tag + "_grad:"):
            close(sample(sd["bb." + key.split(":", 1)[1]].grad, 29), gold[key], rtol=2e-3, atol=1e-5)
            n_grad += 1
    assert n_grad >= 6
    with torch.no_grad():
        close(smp(O.stdcnet813(sd, "bb", x, False, block=block, use_conv_last=last)[4]), gold["%s_eval_feat4" % tag])
