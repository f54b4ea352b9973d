"""ADVENT's entropy / self-information kernels without a GPU: every refusal of the Python layer before any device
call and of the C ABI before any device work, and the resource usage of the compiled csrc/entropy.cu instances."""
import ctypes
import os
import re
import subprocess

import pytest
import torch

from tests.test_classes_cpu import MAX_UPSAMPLE_STACK, _cuobjdump

B200_EINVAL = -1


@pytest.fixture
def no_device_call(monkeypatch):
    from dasemanticsegmentationaml_b200 import _lib
    from dasemanticsegmentationaml_b200 import kernels as K

    def no_call(*a, **k):
        raise AssertionError("no entry point may be called")
    monkeypatch.setattr(_lib, "call", no_call)
    monkeypatch.setattr(K, "call", no_call)


def _lr(n=2, h=16, w=32, ld=32, device="cpu"):
    return torch.zeros((n, h, w, ld), dtype=torch.float32, device=device)


@pytest.mark.parametrize("kw, match", [
    (dict(n_classes=1), "2 to 32"), (dict(n_classes=33), "2 to 32"), (dict(n_classes=19.0), "2 to 32"),
    (dict(n_classes=True), "2 to 32"),
    (dict(lr=_lr(ld=18)), "multiple of 4"), (dict(lr=_lr(ld=16)), ">= 20"),
    (dict(lr=_lr().double()), "fp32"), (dict(lr=_lr()[..., :20]), "contiguous"),
    (dict(H=0), "positive"),
    (dict(lr=_lr(device="meta")), "CUDA tensors"), (dict(lr=_lr()), "CUDA tensors"),
])
@pytest.mark.parametrize("fn", ["upsample_entropy", "upsample_self_information"])
def test_losses_refuse_before_any_device_call(no_device_call, fn, kw, match):
    from dasemanticsegmentationaml_b200 import losses as L
    args = dict(lr=_lr(), H=128, W=256, n_classes=19)
    args.update(kw)
    with pytest.raises(ValueError, match=re.escape(match)):
        getattr(L, fn)(**args)


def test_wrappers_refuse_bad_maps(no_device_call):
    from dasemanticsegmentationaml_b200 import kernels as K
    lr = _lr(device="meta")

    def fwd(emap, layout=K.MAP_PLAIN, H=128, W=256):
        K.entropy_fwd(lr, H, W, 19, K.ENT_MAP, emap=emap, layout=layout)

    bf = dict(dtype=torch.bfloat16, device="meta")
    with pytest.raises(ValueError, match="must be 32 channels"):
        fwd(torch.empty((2, 128, 256, 24), **bf))
    with pytest.raises(ValueError, match="even H and W"):
        fwd(torch.empty((2, 129, 258, 32), **bf), K.MAP_ZERO_BORDERED, H=127)
    with pytest.raises(ValueError, match="even H and W"):
        fwd(torch.empty((2, 130, 257, 32), **bf), K.MAP_ZERO_BORDERED, W=255)
    with pytest.raises(ValueError, match="contiguous bf16"):
        fwd(torch.empty((2, 128, 256, 32), **bf), K.MAP_ZERO_BORDERED)       # the plain shape in layout 2
    with pytest.raises(ValueError, match="contiguous bf16"):
        fwd(torch.empty((2, 128, 256, 32), dtype=torch.float32, device="meta"))
    with pytest.raises(ValueError, match="layout"):
        fwd(torch.empty((2, 128, 256, 32), **bf), 3)
    with pytest.raises(ValueError, match="CUDA tensors"):
        K.entropy_fwd(lr, 128, 256, 19, K.ENT_MAP, emap=torch.empty((2, 128, 256, 32), dtype=torch.bfloat16))
    with pytest.raises(ValueError, match="needs acc"):
        K.entropy_fwd(lr, 128, 256, 19, K.ENT_SUM)
    with pytest.raises(ValueError, match="a map gradient"):
        K.entropy_bwd(lr, 128, 256, 19, K.ENT_SELF_INFO, torch.empty_like(lr))
    with pytest.raises(ValueError, match="d_lr must be"):
        K.entropy_bwd(lr, 128, 256, 19, K.ENT_TRAIN, torch.empty((2, 16, 32, 20), device="meta"))
    with pytest.raises(ValueError, match="CUDA tensors"):
        K.entropy_bwd(lr, 128, 256, 19, K.ENT_TRAIN, torch.empty(lr.shape))


def _abi():
    from dasemanticsegmentationaml_b200 import _lib, build
    if not os.path.exists(build.LIB):
        pytest.skip("the library is not built")
    lib = ctypes.CDLL(build.LIB)
    lib.b200_last_error.restype = ctypes.c_char_p
    return lib, _lib


# (lr_ld, N, h_lr, w_lr, H, W, n_classes, mode, p_ld, layout, message); mode 1 is a map mode of both entry points
ABI_CASES = [
    (32, 2, 16, 32, 128, 256, 1, 0, 32, 1, "classes unsupported"),
    (32, 2, 16, 32, 128, 256, 33, 0, 32, 1, "classes unsupported"),
    (18, 2, 16, 32, 128, 256, 13, 0, 32, 1, "multiple of 4"),
    (12, 2, 16, 32, 128, 256, 13, 0, 32, 1, ">= 16"),
    (32, 2, 16, 32, 128, 256, 19, 1, 24, 1, "map pixel stride 24"),
    (32, 2, 16, 32, 128, 256, 19, 1, 64, 2, "map pixel stride 64"),
    (32, 2, 16, 32, 127, 256, 19, 1, 32, 2, "even H and W"),
    (32, 2, 16, 32, 128, 255, 19, 1, 32, 2, "even H and W"),
    (32, 2, 16, 32, 128, 256, 19, 1, 32, 3, "layout 3"),
    (32, 2, 16, 32, 128, 256, 19, 2, 32, 1, "mode 2"),
    (32, 2, 32, 64, 128, 256, 19, 0, 32, 1, "up-sampling factor"),    # factor 4
    (32, 2, 16, 32, 0, 256, 19, 0, 32, 1, "empty size"),
    (32, 40000, 8, 16, 64, 1024, 19, 0, 32, 1, "exceeds"),           # 2.7e9 pixels with the border
]


@pytest.mark.parametrize("case", ABI_CASES, ids=[c[-1] for c in ABI_CASES])
@pytest.mark.parametrize("entry", ["b200_entropy_fwd", "b200_entropy_bwd"])
def test_abi_refuses_before_device_work(entry, case):
    """NULL data pointers: a refusal must come from the argument checks, before anything touches them."""
    lib, _ = _abi()
    lr_ld, n, h_lr, w_lr, H, W, ncls, mode, p_ld, layout, msg = case
    i = ctypes.c_int
    v = ctypes.c_void_p
    head = (v(0), i(lr_ld), i(n), i(h_lr), i(w_lr), i(H), i(W), i(ncls), i(mode), v(0), i(p_ld), i(layout))
    if entry == "b200_entropy_fwd":
        rc = lib.b200_entropy_fwd(*head, v(0), v(0))
    else:
        rc = lib.b200_entropy_bwd(*head, v(0), v(0), v(0))
    assert rc == B200_EINVAL
    err = lib.b200_last_error().decode()
    assert msg in err, err


def test_abi_requires_its_buffers():
    lib, _ = _abi()
    i = ctypes.c_int
    v = ctypes.c_void_p
    head = lambda mode: (v(0), i(32), i(2), i(16), i(32), i(128), i(256), i(19), i(mode), v(0), i(32), i(1))  # noqa: E731
    assert lib.b200_entropy_fwd(*head(0), v(0), v(0)) == B200_EINVAL
    assert "needs the accumulator" in lib.b200_last_error().decode()
    assert lib.b200_entropy_fwd(*head(1), v(0), v(0)) == B200_EINVAL
    assert "needs the map" in lib.b200_last_error().decode()
    assert lib.b200_entropy_bwd(*head(0), v(0), v(0), v(0)) == B200_EINVAL
    assert "d_lr is required" in lib.b200_last_error().decode()


def test_entropy_instances_resource_usage():
    """Both kernels have an instance per class count 2..32 (62 in all); none needs local memory or more stack
    than the up-sampling family's limit."""
    from dasemanticsegmentationaml_b200 import build
    tool = _cuobjdump()
    if tool is None or not os.path.exists(build.LIB):
        pytest.skip("cuobjdump or the built library is not available")
    r = subprocess.run([tool, "-res-usage", build.LIB], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    usage = {}
    name = None
    for line in r.stdout.splitlines():
        m = re.search(r"Function (_ZN4b200\d+(entropy_\w+?_kernel)ILi(\d+)E\w*):", line)
        if m:
            name = (m.group(2), int(m.group(3)))
            continue
        m = re.search(r"STACK:(\d+) .*LOCAL:(\d+)", line)
        if m and name is not None:
            usage[name] = (int(m.group(1)), int(m.group(2)))
            name = None
    want = [(k, n) for k in ("entropy_fwd_kernel", "entropy_bwd_kernel") for n in range(2, 33)]
    assert sorted(usage) == sorted(want)
    worst = {k: v for k, v in usage.items() if v[0] > MAX_UPSAMPLE_STACK or v[1] > 0}
    assert not worst, worst
