"""CPU-side checks (no GPU): the C-ABI library builds, loads and exports every symbol declared in
include/b200seg.h; the drop-in modules reproduce the reference's state_dict layout (432-entry BiSeNet,
the three discriminators, the shipped GTA5_10_D1.pth key set); host-side geometry of the implicit GEMM."""
import ctypes
import json
import os
import re

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def lib_path():
    from dasemanticsegmentationaml_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(lib_path):
    lib = ctypes.CDLL(lib_path)
    header = open(os.path.join(ROOT, "include", "b200seg.h")).read()
    names = sorted(set(re.findall(r"\b(b200_\w+)\s*\(", header)))
    assert len(names) >= 35
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, missing
    lib.b200_version.restype = ctypes.c_int
    assert lib.b200_version() >= 100
    lib.b200_last_error.restype = ctypes.c_char_p
    assert isinstance(lib.b200_last_error(), bytes)


def test_sass_contains_blackwell_tensor_and_tma_instructions(lib_path):
    import subprocess
    out = subprocess.run(["cuobjdump", "-sass", lib_path], capture_output=True, text=True).stdout
    assert "UTCHMMA" in out or "UTCMMA" in out, "no tcgen05.mma in SASS"
    assert "UTMALDG" in out, "no TMA tensor loads in SASS"
    assert "LDTM" in out, "no TMEM loads in SASS"
    assert "UTMASTG" in out, "no TMA tensor stores in SASS (the conv epilogue's staging tiles)"
    assert "UTCHMMA.2CTA" in out or "2CTA" in out, "no cta_group::2 MMA in SASS"
    assert "FFMA2" in out and "FADD2" in out, "no packed fp32 arithmetic in SASS (BatchNorm column sums of the conv epilogue)"


def test_product_state_dict_layout_matches_reference():
    from dasemanticsegmentationaml_b200.model import (BiSeNet, FCDiscriminator, DepthWiseSepFCDiscriminator,
                                                      DepthWiseSepBNFCDiscriminator)
    layout = json.load(open(os.path.join(GOLD, "state_dict_layout.json")))
    net = BiSeNet("STDCNet813", 19)
    got = [[k, list(v.shape), str(v.dtype)] for k, v in net.state_dict().items()]
    assert got == layout["bisenet"]
    assert len(got) == 432
    assert [n for n, _ in net.named_parameters()] == layout["bisenet_param_names"]
    assert sum(p.numel() for p in net.parameters()) == 11550496
    for name, cls in (("dense", FCDiscriminator), ("dwsep", DepthWiseSepFCDiscriminator),
                      ("dwsep_bn", DepthWiseSepBNFCDiscriminator)):
        got = [[k, list(v.shape), str(v.dtype)] for k, v in cls(19).state_dict().items()]
        assert got == layout["disc_" + name]
    wrapped = torch.nn.DataParallel(DepthWiseSepBNFCDiscriminator(19)).state_dict()
    assert [[k, list(v.shape), str(v.dtype)] for k, v in wrapped.items()] == layout["shipped_D1"]
    wd, nowd, lr_wd, lr_nowd = net.get_params()
    assert len(wd) + len(nowd) + len(lr_wd) + len(lr_nowd) > 0 and len(lr_wd) == 9


def test_modules_refuse_cpu_tensors():
    from dasemanticsegmentationaml_b200 import _lib
    from dasemanticsegmentationaml_b200.model import ConvX
    from dasemanticsegmentationaml_b200 import utils as U
    with pytest.raises(_lib.B200Error):
        ConvX(16, 16)(torch.zeros(1, 16, 8, 8))
    with pytest.raises(_lib.B200Error):
        U.fast_hist(np.zeros(4, dtype=np.int64), np.zeros(4, dtype=np.int64), 19)


def test_dgrad_geometry_matches_conv_transpose():
    """The parity-class decomposition used for stride-2 data gradients, checked on the host against
    torch's conv_transpose arithmetic for one channel."""
    from dasemanticsegmentationaml_b200 import kernels as K
    for (h, w, r, stride, pad) in [(9, 12, 3, 2, 1), (10, 8, 4, 2, 1), (7, 7, 3, 1, 1), (6, 5, 1, 1, 1)]:
        ho = (h + 2 * pad - r) // stride + 1
        wo = (w + 2 * pad - r) // stride + 1
        g = torch.Generator().manual_seed(h * w)
        wt = torch.randn(1, 1, r, r, generator=g, dtype=torch.float64)
        dz = torch.randn(1, 1, ho, wo, generator=g, dtype=torch.float64)
        x = torch.zeros(1, 1, h, w, dtype=torch.float64, requires_grad=True)
        torch.nn.functional.conv2d(x, wt, stride=stride, padding=pad).backward(dz)
        geom = K.dgrad_geometry(h, w, r, r, stride, pad)
        dx = torch.zeros(h, w, dtype=torch.float64)
        for c in geom.classes:
            for i in range(c["Ho"]):
                for j in range(c["Wo"]):
                    acc = 0.0
                    for dh, dw, slab in c["taps"]:
                        a, b = i * geom.in_stride + dh, j * geom.in_stride + dw
                        if 0 <= a < ho and 0 <= b < wo:
                            acc += dz[0, 0, a, b].item() * wt[0, 0, slab // r, slab % r].item()
                    dx[i * geom.out_stride + c["oa"], j * geom.out_stride + c["ob"]] = acc
        assert torch.allclose(dx, x.grad[0, 0], atol=1e-12)


def test_poly_lr_and_per_class_iu_host_side():
    from dasemanticsegmentationaml_b200 import utils as U
    from oracle import segnet_oracle as O
    opt = torch.optim.SGD([torch.nn.Parameter(torch.zeros(1))], lr=0.1)
    assert U.poly_lr_scheduler(opt, 0.01, 3, max_iter=50) == O.poly_lr(0.01, 3, 50)
    assert opt.param_groups[0]["lr"] == O.poly_lr(0.01, 3, 50)
    h = np.arange(361).reshape(19, 19)
    assert np.array_equal(U.per_class_iu(h), O.per_class_iu(h))


def test_ctypes_wrappers_match_header_arity():
    """ctypes sees no prototypes: every `call("b200_*", ...)` site must pass exactly as many positional
    arguments as include/b200seg.h declares (a drift is a corrupted call frame on the GPU box)."""
    import ast
    from dasemanticsegmentationaml_b200 import _lib
    _lib._load_arity()
    assert len(_lib._arity) >= 35
    pkg = os.path.join(ROOT, "dasemanticsegmentationaml_b200")
    seen = set()
    for fname in ("kernels.py", "ops.py"):
        tree = ast.parse(open(os.path.join(pkg, fname)).read())
        for node in ast.walk(tree):
            if isinstance(node, ast.Call) and getattr(node.func, "id", getattr(node.func, "attr", None)) == "call" \
                    and node.args and isinstance(node.args[0], ast.Constant) and str(node.args[0].value).startswith("b200_"):
                name = node.args[0].value
                assert name in _lib._arity, name
                assert len(node.args) - 1 == _lib._arity[name], (fname, name, len(node.args) - 1, _lib._arity[name])
                seen.add(name)
    assert len(seen) >= 30


# Entry points that compute nothing a test could compare: library queries, diagnostics, the NCCL plumbing.
NOT_COMPUTE = {"b200_version", "b200_check_device", "b200_last_error", "b200_optim_chunk",
               "b200_debug_timeline", "b200_debug_knob", "b200_nccl_unique_id", "b200_nccl_init",
               "b200_nccl_allreduce_grads", "b200_nccl_allreduce_hist", "b200_nccl_destroy"}
# Entry points checked exactly through a higher-level call: entry point -> (test file, test, why that suffices).
CHECKED_THROUGH = {
    "b200_image_resize_normalize": ("test_input_gpu.py", "test_reference_dataset_items_bit_exact",
                                    "bit-exact against the reference dataset items through dataset"),
    "b200_label_resize_remap": ("test_input_gpu.py", "test_reference_dataset_items_bit_exact",
                                "bit-exact against the reference dataset labels through dataset"),
    "b200_count_equal": ("test_modules_gpu.py", "test_eval_metric_bit_exact",
                         "utils.compute_global_accuracy equals the oracle's exactly"),
    "b200_wgrad_unscratch_pairview": ("test_modules_gpu.py", "test_dense_discriminator_pair_view",
                                      "the pair-view weight gradient is compared with torch's"),
    "b200_upsample_fwd": ("test_modules_gpu.py", "test_fused_losses_against_torch",
                          "every mode through losses.py against F.interpolate + torch's losses"),
    "b200_upsample_bwd": ("test_modules_gpu.py", "test_fused_losses_against_torch",
                          "every mode's gradient through losses.py against torch autograd"),
    "b200_sgd_step": ("test_blocks_gpu.py", "test_fused_optimizers_match_torch",
                      "optim.py's fused step against torch.optim.SGD"),
    "b200_adam_step": ("test_blocks_gpu.py", "test_fused_optimizers_match_torch",
                       "optim.py's fused step against torch.optim.Adam"),
}


def test_every_compute_entry_point_has_a_direct_gpu_test():
    """Every compute entry point of include/b200seg.h is named in some tests/*_gpu.py, as its b200_ symbol or as
    `K.<wrapper>(` of its kernels.py wrapper, or is listed above with the test that checks it -- so a new kernel
    cannot land without a direct test."""
    import ast
    import glob
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "b200seg.h")).read(), flags=re.S)
    names = sorted(set(re.findall(r"\b(b200_\w+)\s*\(", header)))
    assert len(names) >= 35
    wrappers = {}
    tree = ast.parse(open(os.path.join(ROOT, "dasemanticsegmentationaml_b200", "kernels.py")).read())
    for fn in tree.body:
        if isinstance(fn, ast.FunctionDef):
            for node in ast.walk(fn):
                if isinstance(node, ast.Constant) and isinstance(node.value, str) and node.value.startswith("b200_"):
                    wrappers.setdefault(node.value, set()).add(fn.name)
    tests = {os.path.basename(p): open(p).read() for p in glob.glob(os.path.join(ROOT, "tests", "*_gpu.py"))}
    text = "\n".join(tests.values())
    for name, (fname, test, why) in CHECKED_THROUGH.items():
        assert name in names, "allow-listed entry point %s is not declared" % name
        assert "def %s(" % test in tests.get(fname, ""), "%s: %s::%s does not exist" % (name, fname, test)
    untested = [n for n in names if n not in NOT_COMPUTE and n not in CHECKED_THROUGH and n not in text
                and not any("K.%s(" % w in text for w in wrappers.get(n, ()))]
    assert not untested, "entry points without a direct GPU test: %s" % untested


def test_checkpoint_helpers_round_trip(tmp_path):
    """train.py:110,118,282-283: seg-net files carry bare keys, discriminator files `module.`-prefixed
    ones (the shipped GTA5_10_D1.pth); both must load into bare and wrapped modules."""
    from dasemanticsegmentationaml_b200 import checkpoint as C
    from dasemanticsegmentationaml_b200.model import DepthWiseSepBNFCDiscriminator
    torch.manual_seed(3)
    a, b = DepthWiseSepBNFCDiscriminator(19), DepthWiseSepBNFCDiscriminator(19)
    path = C.save_state(a, str(tmp_path / "ckpt" / "GTA5_10_D1.pth"), keep_wrapper_prefix=True)
    saved = torch.load(path)
    with open(os.path.join(GOLD, "state_dict_layout.json")) as f:
        shipped = json.load(f)["shipped_D1"]
    assert [(k, list(v.shape)) for k, v in saved.items()] == [(k, s) for k, s, _ in shipped]
    assert C.load_state(b, path) == []
    for (k, v), (_, w) in zip(a.state_dict().items(), b.state_dict().items()):
        assert torch.equal(v, w), k
    # bare keys, wrapped target, partial overlay (BiSeNet.load_weight semantics); DataParallel moves the
    # module to cuda:0 when a GPU is present, so the loaded values are compared on the host
    wrapped = torch.nn.DataParallel(DepthWiseSepBNFCDiscriminator(19))
    partial = {k: v for k, v in a.state_dict().items() if k.startswith("conv1_d")}
    assert partial
    partial["not.a.key"] = torch.zeros(1)
    assert C.load_state(wrapped, partial, strict=False) == ["not.a.key"]
    for k, v in partial.items():
        if k != "not.a.key":
            assert torch.equal(wrapped.module.state_dict()[k].cpu(), v), k


def test_input_tables_match_oracle():
    """Host side of the input pipeline: the vectorised table builders against the oracle's scalar
    restatement of Pillow, at the dataset sizes and a few odd ones."""
    from dasemanticsegmentationaml_b200 import dataset as D
    from oracle import input_oracle as I
    for (i, o) in [(96, 48), (97, 50), (50, 100), (1914, 512), (1052, 1024), (2048, 1280), (1024, 720), (33, 33)]:
        b, k = D.bilinear_tables(i, o)
        xmin, cnt, kk = I.bilinear_coeffs(i, o)
        assert np.array_equal(b[:, 0], xmin) and np.array_equal(b[:, 1], cnt) and np.array_equal(k, kk)
        assert np.array_equal(D.nearest_table(i, o), I.nearest_index(i, o))
    ref = I.to_tensor_normalize(np.arange(256, dtype=np.uint8)[None, :, None].repeat(3, 2))[:, 0]
    assert np.array_equal(D.normalize_table().numpy(), ref)
    lut = D.label_table(D.GTA5_ID_TO_TRAINID).numpy()
    ids = np.arange(256, dtype=np.uint8)
    assert np.array_equal(lut, I.convert_labels(ids, {k: v for k, v in D.GTA5_ID_TO_TRAINID.items() if k >= 0}))


def test_dataset_classes_discover_and_decode_like_the_reference(tmp_path):
    """Host half of the input pipeline (no GPU): directory layouts, sorting / pairing, the 'color'
    label files being skipped (cityscapes.py:37-57), decoded uint8 items, collate_raw, aug_type."""
    from PIL import Image
    from dasemanticsegmentationaml_b200 import dataset as D
    rng = np.random.default_rng(1)
    cs = tmp_path / "cs"
    want = {}
    for city, names in (("bern", ["b_2", "b_1"]), ("aachen", ["a_1"])):
        (cs / "images" / "train" / city).mkdir(parents=True)
        (cs / "gtFine" / "train" / city).mkdir(parents=True)
        for nm in names:
            img = rng.integers(0, 256, (20, 30, 3), dtype=np.uint8)
            lab = rng.integers(0, 19, (20, 30), dtype=np.uint8)
            Image.fromarray(img).save(str(cs / "images" / "train" / city / (nm + "_leftImg8bit.png")))
            Image.fromarray(lab).save(str(cs / "gtFine" / "train" / city / (nm + "_gtFine_labelTrainIds.png")))
            Image.fromarray(img).save(str(cs / "gtFine" / "train" / city / (nm + "_gtFine_color.png")))
            want[nm] = (img, lab)
    (cs / "images" / "train" / "notes.txt").write_text("not a city")
    ds = D.CityScapes("train", str(cs), 16, 32)
    assert len(ds) == 3
    order = [os.path.basename(p).split("_leftImg8bit")[0] for p, _ in ds.data]
    assert order == ["a_1", "b_1", "b_2"]                      # sorted full paths, as the reference pairs them
    for i, nm in enumerate(order):
        assert nm in os.path.basename(ds.data[i][1])
        img, lab = ds[i]
        assert img.dtype == torch.uint8 and lab.dtype == torch.uint8
        assert np.array_equal(img.numpy(), want[nm][0]) and np.array_equal(lab.numpy(), want[nm][1])
    imgs, labs = D.collate_raw([ds[0], ds[1]])
    assert imgs.shape == (2, 20, 30, 3) and labs.shape == (2, 20, 30)
    other = (torch.zeros(10, 12, 3, dtype=torch.uint8), torch.zeros(10, 12, dtype=torch.uint8))
    imgs, labs = D.collate_raw([ds[0], other])
    assert isinstance(imgs, list) and len(labs) == 2            # mixed source sizes stay a list
    assert (ds.preprocess.out_w, ds.preprocess.out_h) == (16, 32)   # the reference's (height, width) -> PIL (w, h)
    gta = tmp_path / "gta"
    (gta / "images").mkdir(parents=True)
    (gta / "labels").mkdir()
    Image.fromarray(want["a_1"][0]).save(str(gta / "images" / "00001.png"))
    Image.fromarray(want["a_1"][1]).save(str(gta / "labels" / "00001.png"))
    g = D.GtaV(str(gta), None, 16, 32)
    assert len(g) == 1 and g.lb_map[7] == 0 and g.lb_map[33] == 18 and g.lb_map[0] == 255
    assert torch.equal(g.convert_labels(torch.tensor([7, 0, 33, 200], dtype=torch.uint8)),
                       torch.tensor([0, 255, 18, 200], dtype=torch.uint8))
    with pytest.raises(NotImplementedError):
        D.GtaV(str(gta), "H-RP", 16, 32)


def test_fused_optimizers_refuse_cpu_parameters():
    from dasemanticsegmentationaml_b200 import optim as B200Optim
    from dasemanticsegmentationaml_b200._lib import B200Error
    p = torch.nn.Parameter(torch.ones(4))
    p.grad = torch.ones(4)
    for opt in (B200Optim.FusedSGD([p], lr=0.1, momentum=0.9), B200Optim.FusedAdam([p], lr=0.1)):
        with pytest.raises(B200Error):
            opt.step()
    with pytest.raises(ValueError):
        B200Optim.FusedSGD([p], lr=0.1, nesterov=True)

def test_tuned_tile_table_is_well_formed():
    """dasemanticsegmentationaml_b200/tuned_tiles.json: every entry parses back into a launch the C launcher accepts by
    construction (the GPU suite, tests/test_tuned_gpu.py, then checks each one numerically)."""
    import re
    path = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "dasemanticsegmentationaml_b200",
                        "tuned_tiles.json")
    table = json.load(open(path))
    assert len(table) >= 100
    for key, word in table.items():
        assert isinstance(word, int) and 0 < word < (1 << 31), key
        if key.startswith("conv "):
            m = re.match(r"conv (\d+) (\d+) (\d+) c(\d+) r(\d+) (\S+)( f32)?( st)?( mk)?$", key)
            assert m, key
            rows, bn = int(m.group(5)), word & 0xFFF
            assert bn in (16, 32, 64, 128, 256) and rows % bn == 0, (key, bn)
            pair, persistent, halo = (word >> 22) & 1, (word >> 20) & 1, (word >> 23) & 1
            assert not (pair and persistent), key
            assert not halo or pair, key                       # halo rings exist in the CTA-pair kernel only
            if pair:
                assert bn >= 32, key
            assert not ((word >> 27) & 1 and (word >> 28) & 1), key   # register stores XOR forced TMA stores
            assert not (m.group(7) and (word >> 28) & 1), key          # fp32 outputs never leave through TMA stores
        else:
            m = re.match(r"wgrad (\d+) (\d+) (\d+) co(\d+) ci(\d+) (\d+)x(\d+)s(\d+)$", key)
            assert m, key
            assert (word & 0xFFF) in (64, 128, 192, 256), key
            assert 0 <= ((word >> 12) & 0xF) <= 8 and ((word >> 28) & 3) in (0, 1, 2), key
