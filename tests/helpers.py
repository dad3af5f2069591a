"""Shared helpers for the parity tests."""
import torch

from oracle import genie_oracle as O


def det_weights(module, gain=1.0):
    """Closed-form weights (the same ones oracle/make_golden.py loaded into the reference)."""
    shapes = {k: tuple(v.shape) for k, v in module.state_dict().items()}
    sd = O.det_state_dict(shapes, gain)
    missing = module.load_state_dict(sd, strict=False)
    assert all(k.endswith(('freq', 'bit_mask', 'blur')) for k in missing.missing_keys), missing
    return {k: v.detach().clone().cpu() for k, v in module.state_dict().items()}


def at_sample(t, key, ref):
    """`t` (reference layout) on the deterministic sample that the golden `ref` stores (genie_oracle.det_sample)."""
    return O.det_sample(t.detach().float(), key, ref.numel()).cpu()


def bf16_round(t):
    return t.to(torch.bfloat16).to(torch.float32)


def round_conv_weights(sd):
    """What the kernels see: conv / 5-D weights rounded to bf16, everything else fp32."""
    return {k: (bf16_round(v) if v.dim() == 5 else v) for k, v in sd.items()}


def rel_l2(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return ((a - b).norm() / b.norm().clamp_min(1e-30)).item()


def assert_close(got, ref, rtol, atol, name=''):
    got, ref = got.detach().float().cpu(), ref.detach().float().cpu()
    assert got.shape == ref.shape, f'{name}: shape {tuple(got.shape)} vs {tuple(ref.shape)}'
    err = (got - ref).abs()
    bad = err > atol + rtol * ref.abs()
    if bad.any():
        i = torch.nonzero(bad.flatten())[0].item()
        raise AssertionError(f'{name}: {int(bad.sum())}/{bad.numel()} mismatches (rtol={rtol}, atol={atol}); '
                             f'max err {err.max().item():.3e}; first at flat {i}: got {got.flatten()[i].item():.6f} '
                             f'ref {ref.flatten()[i].item():.6f}')
