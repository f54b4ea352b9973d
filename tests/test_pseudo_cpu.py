"""Pseudo-labels without a GPU: every request check of train.predict_confidence / pseudo_label_thresholds /
pseudo_labels is made before any device call, and the resource usage of the compiled csrc/pseudo.cu and
msc_confidence kernels."""
import os
import re
import subprocess

import pytest
import torch

from tests.test_classes_cpu import MAX_UPSAMPLE_STACK, _cuobjdump
from tests.test_tta_cpu import _NoForward


@pytest.fixture
def no_device_call(monkeypatch):
    from dasemanticsegmentationaml_b200 import _lib

    def no_call(*a, **k):
        raise AssertionError("no entry point may be called")
    monkeypatch.setattr(_lib, "call", no_call)


@pytest.mark.parametrize("n, hw, scales, flip, match", [
    (2, (512, 1024), (), False, "at least one"),
    (2, (512, 1024), (1.0, 0.0), False, "> 0"),
    (2, (512, 1024), (float("nan"),), False, "> 0"),
    (2, (512, 1024), (0.12,), False, ">= 64"),
    (2, (512, 1024), (0.5,) * 9, True, "at most 16"),
    (33, (256, 512), (1.0,), True, "2N = 66"),
])
def test_predict_confidence_refuses_before_any_device_call(no_device_call, n, hw, scales, flip, match):
    from dasemanticsegmentationaml_b200 import train as T
    images = torch.empty((n, 3) + hw, device="meta")
    with pytest.raises(ValueError, match=re.escape(match)):
        T.predict_confidence(_NoForward(), images, scales=scales, flip=flip)


def _batch(shape=(2, 8, 8), pred_dtype=torch.uint8, conf_dtype=torch.float32):
    return torch.empty(shape, dtype=pred_dtype, device="meta"), torch.empty(shape, dtype=conf_dtype, device="meta")


@pytest.mark.parametrize("kw, match", [
    (dict(portion=0.0), "portion"), (dict(portion=-0.5), "portion"), (dict(portion=1.5), "portion"),
    (dict(portion=float("nan")), "portion"), (dict(portion=float("inf")), "portion"), (dict(portion="0.5"), "portion"),
    (dict(cap=0.0), "cap"), (dict(cap=1.01), "cap"), (dict(cap=float("nan")), "cap"), (dict(cap=-float("inf")), "cap"),
    (dict(n_classes=1), "2 to 32"), (dict(n_classes=33), "2 to 32"), (dict(n_classes=19.0), "2 to 32"),
])
def test_thresholds_refuse_bad_parameters(no_device_call, kw, match):
    from dasemanticsegmentationaml_b200 import train as T
    p, c = _batch()
    with pytest.raises(ValueError, match=re.escape(match)):
        T.pseudo_label_thresholds([p], [c], **kw)


def test_thresholds_refuse_mismatched_lists(no_device_call):
    from dasemanticsegmentationaml_b200 import train as T
    p, c = _batch()
    with pytest.raises(ValueError, match="equal, non-zero length"):
        T.pseudo_label_thresholds([p, p], [c])
    with pytest.raises(ValueError, match="equal, non-zero length"):
        T.pseudo_label_thresholds([], [])
    p2, c2 = _batch((2, 8, 9))
    with pytest.raises(ValueError, match="batch 1"):
        T.pseudo_label_thresholds([p, p], [c, c2])
    with pytest.raises(ValueError, match="batch 0"):
        T.pseudo_label_thresholds(*[[t] for t in _batch(pred_dtype=torch.int64)])
    with pytest.raises(ValueError, match="batch 0"):
        T.pseudo_label_thresholds(*[[t] for t in _batch(conf_dtype=torch.float16)])


def test_labels_refuse_bad_requests(no_device_call):
    from dasemanticsegmentationaml_b200 import train as T
    p, c = _batch()
    for bad in (float("nan"), float("inf"), "0.9", None):
        with pytest.raises(ValueError, match="global threshold"):
            T.pseudo_labels(p, c, bad)
    for shape in ((1,), (33,), (2, 19)):
        with pytest.raises(ValueError, match="thresholds"):
            T.pseudo_labels(p, c, torch.empty(shape, device="meta"))
    with pytest.raises(ValueError, match="dtype"):
        T.pseudo_labels(p, c, 0.9, dtype=torch.int32)
    p2, _ = _batch((2, 8, 9))
    with pytest.raises(ValueError, match="one shape"):
        T.pseudo_labels(p2, c, 0.9)


def test_pseudo_instances_resource_usage():
    """msc_confidence has an instance per class count 2..32 and the three selection kernels are present; none
    needs more stack than the up-sampling family's limit or any local memory."""
    from dasemanticsegmentationaml_b200 import build
    tool = _cuobjdump()
    if tool is None or not os.path.exists(build.LIB):
        pytest.skip("cuobjdump or the built library is not available")
    r = subprocess.run([tool, "-res-usage", build.LIB], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    kernels = "msc_confidence_kernel|class_select_hist_kernel|class_select_pick_kernel|pseudo_label_apply_kernel"
    usage = {}
    name = None
    for line in r.stdout.splitlines():
        m = re.search(r"Function (_ZN4b200\d+(%s)(?:ILi(\d+)E)?\w*):" % kernels, line)
        if m:
            name = (m.group(2), int(m.group(3)) if m.group(3) else None)
            continue
        m = re.search(r"STACK:(\d+) .*LOCAL:(\d+)", line)
        if m and name is not None:
            usage[name] = (int(m.group(1)), int(m.group(2)))
            name = None
    want = [("msc_confidence_kernel", n) for n in range(2, 33)] + [
        ("class_select_hist_kernel", None), ("class_select_pick_kernel", None), ("pseudo_label_apply_kernel", None)]
    missing = [k for k in want if k not in usage]
    assert not missing, missing
    worst = {k: v for k, v in usage.items() if v[0] > MAX_UPSAMPLE_STACK or v[1] > 0}
    assert not worst, worst
