"""Multi-scale + flip evaluation without a GPU: the request checks of train.predict, and the resource usage of
the compiled csrc/msc.cu kernels."""
import os
import re
import subprocess

import pytest
import torch

from tests.test_classes_cpu import MAX_UPSAMPLE_STACK, _cuobjdump


class _NoForward(object):
    n_classes = 19

    def eval(self):
        raise AssertionError("the request must be refused before the model is touched")

    def forward_lowres(self, x):
        raise AssertionError("the request must be refused before any forward")


@pytest.mark.parametrize("n, hw, scales, flip, match", [
    (2, (512, 1024), (), False, "at least one"),
    (2, (512, 1024), (1.0, 0.0), False, "> 0"),
    (2, (512, 1024), (-0.5,), True, "> 0"),
    (2, (512, 1024), (float("nan"),), False, "> 0"),
    (2, (512, 1024), (float("inf"),), False, "> 0"),
    (2, (512, 1024), (0.12,), False, ">= 64"),       # 61 x 122
    (1, (64, 2048), (1.0, 0.99), True, ">= 64"),     # 63 rows
    (2, (512, 1024), (0.5,) * 9, True, "at most 16"),
    (2, (512, 1024), (0.5,) * 17, False, "at most 16"),
    (33, (256, 512), (1.0,), True, "2N = 66"),
])
def test_predict_refuses_before_any_device_call(monkeypatch, n, hw, scales, flip, match):
    from dasemanticsegmentationaml_b200 import _lib
    from dasemanticsegmentationaml_b200 import train as T

    def no_call(*a, **k):
        raise AssertionError("no entry point may be called")
    monkeypatch.setattr(_lib, "call", no_call)
    images = torch.empty((n, 3) + hw, device="meta")
    with pytest.raises(ValueError, match=re.escape(match)):
        T.predict(_NoForward(), images, scales=scales, flip=flip)


def test_predict_limits_accept_the_edges():
    from dasemanticsegmentationaml_b200 import train as T
    images = torch.empty((32, 3, 512, 1024), device="meta")
    assert T._tta_sizes(images, (0.125,) * 8, True) == [(64, 128)] * 8
    assert T._tta_sizes(images, (0.5, 0.75, 1.0, 1.25, 1.5, 1.75), False)[-1] == (896, 1792)
    assert T._tta_sizes(torch.empty((1, 3, 720, 1280), device="meta"), (0.6,), False) == [(432, 768)]


def test_msc_instances_resource_usage():
    """Every class count 2..32 has its combine instance and the rescale kernel is present; none needs more
    stack than the up-sampling family's limit or any local memory."""
    from dasemanticsegmentationaml_b200 import build
    tool = _cuobjdump()
    if tool is None or not os.path.exists(build.LIB):
        pytest.skip("cuobjdump or the built library is not available")
    r = subprocess.run([tool, "-res-usage", build.LIB], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    usage = {}
    name = None
    for line in r.stdout.splitlines():
        m = re.search(r"Function (_ZN4b200\d+(msc_argmax_kernel|image_rescale_kernel)(?:ILi(\d+)E)?\w*):", line)
        if m:
            name = (m.group(2), int(m.group(3)) if m.group(3) else None)
            continue
        m = re.search(r"STACK:(\d+) .*LOCAL:(\d+)", line)
        if m and name is not None:
            usage[name] = (int(m.group(1)), int(m.group(2)))
            name = None
    want = [("msc_argmax_kernel", n) for n in range(2, 33)] + [("image_rescale_kernel", None)]
    missing = [k for k in want if k not in usage]
    assert not missing, missing
    worst = {k: v for k, v in usage.items() if v[0] > MAX_UPSAMPLE_STACK or v[1] > 0}
    assert not worst, worst
