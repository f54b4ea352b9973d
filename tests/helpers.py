import numpy as np
import torch


def rel_l2(a, b):
    a, b = a.detach().float().cpu(), b.detach().float().cpu()
    return ((a - b).norm() / (b.norm() + 1e-20)).item()


def cosine(a, b):
    a, b = a.detach().float().cpu().reshape(-1), b.detach().float().cpu().reshape(-1)
    return (torch.dot(a, b) / (a.norm() * b.norm() + 1e-30)).item()


def bf16_round(t):
    return t.to(torch.bfloat16).float()


def load_oracle_state(module, sd, prefix=""):
    """Copies an oracle state dict (no alias keys) into a product module."""
    own = module.state_dict()
    for k, v in sd.items():
        if not k.startswith(prefix):
            continue
        kk = k[len(prefix):]
        assert kk in own and own[kk].shape == v.shape, kk
        own[kk] = v.detach().clone()
    module.load_state_dict(own)
    return module


def sub_state(sd, prefix):
    return {k: v for k, v in sd.items() if k.startswith(prefix)}


def to_device(sd, device, requires_grad=False):
    out = {}
    for k, v in sd.items():
        t = v.detach().clone().to(device)
        if requires_grad and t.is_floating_point() and "running_" not in k:
            t.requires_grad_(True)
        out[k] = t
    return out


def gate(name, value, threshold):
    """Assert value > threshold, printing the measured number so that a GPU run's log records it."""
    print("GATE %-60s %.6f (> %.4f)" % (name, value, threshold))
    assert value > threshold, (name, value, threshold)


# Element-wise gates of the direct kernel tests (test_norm_gpu, test_attention_gpu, test_heads_losses_gpu):
# a kernel output against a float64 reference computed from the same bf16-rounded inputs.
def bf16_ulp(ref):
    """One bf16 ulp at |ref| (8 significant bits), float64."""
    e = torch.frexp(ref.abs().clamp_min(2.0 ** -126))[1]
    return torch.ldexp(torch.ones_like(ref, dtype=torch.float64), e - 8)


def assert_within(name, got, want, tol, skip=None):
    err = (got.double() - want.double()).abs()
    ok = err <= tol
    if skip is not None:
        ok = ok | skip
    worst = (err / tol).max().item() if err.numel() else 0.0
    print("%-44s max err/tol %.3f" % (name, worst))
    if not bool(ok.all()):
        i = int((~ok).reshape(-1).nonzero()[0])
        raise AssertionError("%s: %d elements out of bound; first at flat %d: got %r want %r tol %r" % (
            name, int((~ok).sum()), i, got.reshape(-1)[i].item(), want.reshape(-1)[i].item(),
            tol.reshape(-1)[i].item() if torch.is_tensor(tol) and tol.numel() > 1 else float(tol)))


def assert_bf16(name, got, want, terms=None, skip=None):
    tol = bf16_ulp(want)
    if terms is not None:
        tol = tol + 1e-4 * terms
    assert_within(name, got, want, tol, skip)


def assert_f32_sum(name, got, want, abs_terms):
    assert_within(name, got, want, 1e-5 * abs_terms.double() + 1e-6)


class quantised_oracle(object):
    """Context manager: oracle stores conv outputs / activations as bf16 like the CUDA path
    (SURVEY 8c quantisation-matched oracle)."""

    def __enter__(self):
        from oracle import segnet_oracle as O
        self._old, O.QUANT = O.QUANT, True

    def __exit__(self, *a):
        from oracle import segnet_oracle as O
        O.QUANT = self._old
