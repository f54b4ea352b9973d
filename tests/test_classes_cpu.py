"""Class counts other than 19 without a GPU: construction limits, state_dict layouts against the oracle, and
the resource usage of the compiled up-sampling instances."""
import os
import re
import shutil
import subprocess

import pytest
import torch

from oracle import segnet_oracle as O

# Local memory (stack frame, bytes) of the 19-class strip backward before the instances were generalised:
# 8 bytes of spill.  No instance of the up-sampling family may need more.
MAX_UPSAMPLE_STACK = 8


@pytest.mark.parametrize("n_classes", [1, 33, 0, 19.0])
def test_unsupported_class_counts_are_refused(n_classes):
    from dasemanticsegmentationaml_b200.model import BiSeNet, BiSeNetOutput
    with pytest.raises(ValueError, match="2 to 32"):
        BiSeNet("STDCNet813", n_classes)
    with pytest.raises(ValueError, match="2 to 32"):
        BiSeNetOutput(64, 64, n_classes)


def _shapes(sd):
    return {k: tuple(v.shape) for k, v in sd.items()}


def test_bisenet_state_dict_matches_oracle_16():
    from dasemanticsegmentationaml_b200.model import BiSeNet
    m = BiSeNet("STDCNet813", 16)
    assert m.n_classes == 16
    want = _shapes(O.make_bisenet_state(n_classes=16))
    got = _shapes(m.state_dict())
    assert set(want) <= set(got)
    assert {k: got[k] for k in want} == want
    # keys the oracle does not build are the backbone's unused ImageNet head; none of them depends on the count
    assert all(not k.endswith("conv_out.weight") for k in set(got) - set(want))
    assert got["conv_out.conv_out.weight"] == (16, 256, 1, 1)


@pytest.mark.parametrize("kind", ["dense", "dwsep", "dwsep_bn"])
def test_discriminator_state_dict_matches_oracle_16(kind):
    from dasemanticsegmentationaml_b200.model import (FCDiscriminator, DepthWiseSepFCDiscriminator,
                                                      DepthWiseSepBNFCDiscriminator)
    cls = {"dense": FCDiscriminator, "dwsep": DepthWiseSepFCDiscriminator, "dwsep_bn": DepthWiseSepBNFCDiscriminator}[kind]
    got = _shapes(cls(16).state_dict())
    want = _shapes(O.make_discriminator_state(kind, n_classes=16))
    assert got == want


def _cuobjdump():
    from dasemanticsegmentationaml_b200 import build
    for cand in (os.path.join(os.path.dirname(build._nvcc()), "cuobjdump"), shutil.which("cuobjdump"),
                 "/usr/local/cuda/bin/cuobjdump"):
        if cand and os.path.isabs(cand) and os.path.exists(cand):
            return cand
    return None


def test_upsample_instances_resource_usage():
    """Every class count 2..32 has its four instances in the library, and none needs more local memory
    (register spill) than the 19-class strip kernel did."""
    from dasemanticsegmentationaml_b200 import build
    tool = _cuobjdump()
    if tool is None or not os.path.exists(build.LIB):
        pytest.skip("cuobjdump or the built library is not available")
    r = subprocess.run([tool, "-res-usage", build.LIB], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    usage = {}
    name = None
    for line in r.stdout.splitlines():
        m = re.search(r"Function (_ZN4b200\d+(upsample_\w+?_kernel)ILi(\d+)E\w*):", line)
        if m:
            name = (m.group(2), int(m.group(3)))
            continue
        m = re.search(r"STACK:(\d+) .*LOCAL:(\d+)", line)
        if m and name is not None:
            usage[name] = (int(m.group(1)), int(m.group(2)))
            name = None
    kernels = ("upsample_fwd_kernel", "upsample_fwd_tiled_kernel", "upsample_bwd_kernel", "upsample_bwd_strip_kernel")
    missing = [(k, n) for k in kernels for n in range(2, 33) if (k, n) not in usage]
    assert not missing, missing
    worst = {k: v for k, v in usage.items() if v[0] > MAX_UPSAMPLE_STACK or v[1] > 0}
    assert not worst, worst
