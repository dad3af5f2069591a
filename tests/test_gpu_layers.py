"""GPU parity tests, layer level: CUDA path (through the C ABI) vs the oracle and the golden vectors.

Tolerances (SURVEY.md §7 H3): both sides consume identical bf16-rounded inputs and conv weights.
  * a single kernel with fp32 output (conv, LFQ, statistics) is gated at rtol=1e-3 / atol=1e-5 (the
    north_star figure) relative to unit-scale data (atol scaled by the reference's magnitude);
  * anything that stores a bf16 tensor is gated at one bf16 ulp on that tensor: rtol=2^-7, plus an atol of
    2^-7 of the tensor's scale.
"""
import pytest
import torch

from helpers import assert_close, at_sample, bf16_round, det_weights, rel_l2, round_conv_weights
from oracle import genie_oracle as O

pytestmark = pytest.mark.gpu
DEV = 'cuda'
BF16_ULP = 2.0 ** -7


def _grads(module):
    return {k: p.grad.detach().float().cpu() for k, p in module.named_parameters() if p.grad is not None}


def _run_layer(layer, x, *extra, wants_f32=False):
    """Forward + backward of mean(y^2) through the CUDA path. Returns y (NCDHW fp32), dx, param grads."""
    from open_genie_b200 import ops
    xg = x.clone().to(DEV).requires_grad_(True)
    y = layer(xg, *extra)
    yr = ops.to_reference(y)
    # d/dy mean(y^2) = 2 y / numel, fed as an explicit upstream gradient
    g = (2.0 / y.numel()) * y.detach().float()
    y.backward(g.to(y.dtype))
    return yr.cpu(), xg.grad.float().cpu(), _grads(layer)


def test_causal_conv3d_matches_golden_and_oracle(golden):
    from open_genie_b200.module.video import CausalConv3d
    g = golden('layers.pt')['causal_conv3d']
    m = CausalConv3d(64, 64, 3)
    sd = det_weights(m)
    m.to(DEV)
    m.out_f32 = True
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    y, dx, grads = _run_layer(m, x)
    sdr = round_conv_weights(sd)
    xr = x.clone().requires_grad_(True)
    w = sdr['conv3d.weight'].clone().requires_grad_(True)
    b = sdr['conv3d.bias'].clone().requires_grad_(True)
    yo = O.causal_conv3d(xr, w, b)
    # single kernel, fp32 out: the north_star tolerance
    assert_close(y, yo, 1e-3, 1e-5 * yo.abs().max().item(), 'conv fwd vs oracle (bf16-rounded operands)')
    # golden was produced by the reference with UNrounded weights/inputs: bf16 operand rounding only
    assert rel_l2(at_sample(y, 'layers.causal_conv3d.y', g['y']), g['y']) < 1e-2
    # backward: upstream gradient is rounded to bf16 by the product; emulate
    gy = bf16_round((2.0 / yo.numel()) * y)
    yo.backward(gy)
    assert_close(dx, xr.grad, BF16_ULP, BF16_ULP * xr.grad.abs().max().item(), 'conv dgrad')
    assert_close(grads['conv3d.weight'], w.grad, 2e-3, 1e-3 * w.grad.abs().max().item(), 'conv wgrad')
    assert_close(grads['conv3d.bias'], b.grad, 2e-3, 1e-3 * b.grad.abs().max().item(), 'conv bias grad')


@pytest.mark.parametrize('cin,cout,stride,shape', [
    (128, 128, (1, 2, 2), (2, 128, 4, 16, 16)),      # enc downsample #1 geometry (time stride 1)
    (256, 256, (2, 2, 2), (2, 256, 4, 8, 8)),        # enc downsample #2/#3 geometry
    (64, 192, (2, 2, 2), (1, 64, 5, 9, 7)),          # ragged extents: partial boxes, odd sizes, Cout != Cin
    (64, 64, (1, 4, 4), (1, 64, 2, 16, 16)),         # stride 4 > kernel 3: residue classes without taps (zero rows of dx)
])
def test_strided_causal_conv_implicit_gemm(cin, cout, stride, shape):
    """SpaceTimeDownsample as an IMPLICIT GEMM (strided TMA boxes forward / wgrad, residue-class data gradient):
    forward, dx and dW against the oracle's F.pad + conv3d on identical bf16-rounded operands."""
    from open_genie_b200.module.video import SpaceTimeDownsample
    from open_genie_b200 import _lib
    m = SpaceTimeDownsample(cin, 3, cout, time_factor=stride[0], space_factor=stride[1])
    assert m.go_down.conv3d.geom.strided_implicit
    sd = det_weights(m)
    m.to(DEV)
    m.go_down.out_f32 = True
    x = bf16_round(O.det_uniform('strided.x', shape))
    _lib.TIMING = []
    try:
        y, dx, grads = _run_layer(m, x)
        names = {t[0] for t in _lib.TIMING}
    finally:
        _lib.TIMING = None
    assert 'og_conv3d_strided_fwd' in names and 'og_conv3d_strided_dgrad' in names and 'og_conv3d_strided_wgrad' in names
    assert not any('im2col' in n or 'col2im' in n for n in names)
    sdr = round_conv_weights(sd)
    xr = x.clone().requires_grad_(True)
    w = sdr['go_down.conv3d.weight'].clone().requires_grad_(True)
    yo = O.causal_conv3d(xr, w, sdr['go_down.conv3d.bias'], stride=stride)
    assert y.shape == yo.shape
    assert_close(y, yo, 1e-3, 1e-5 * yo.abs().max().item(), 'strided implicit fwd')
    yo.backward(bf16_round((2.0 / yo.numel()) * y))
    assert_close(dx, xr.grad, BF16_ULP, BF16_ULP * xr.grad.abs().max().item(), 'strided implicit dgrad')
    assert_close(grads['go_down.conv3d.weight'], w.grad, 2e-3, 1e-3 * w.grad.abs().max().item(), 'strided implicit wgrad')


@pytest.mark.parametrize('cin,cout,stride,shape', [
    (3, 128, (1, 1, 1), (2, 3, 4, 16, 16)),          # tokenizer / LatentAction stem: 3 -> C
    (18, 64, (1, 1, 1), (2, 18, 2, 8, 8)),           # decoder stem: 18 -> C (its input needs a gradient: LFQ backward)
    (3, 64, (1, 4, 4), (1, 3, 2, 16, 16)),           # REPR_TOK_ENC: strided AND narrow
])
def test_narrow_cin_conv_is_an_implicit_gemm_on_padded_channels(cin, cout, stride, shape):
    from open_genie_b200.module.video import CausalConv3d
    from open_genie_b200 import _lib
    m = CausalConv3d(cin, cout, 3, stride=stride)
    g = m.conv3d.geom
    assert g.padded and g.cin_pad == 64 and (g.direct or g.strided_implicit)
    sd = det_weights(m)
    m.to(DEV)
    m.out_f32 = True
    x = bf16_round(O.det_uniform('narrow.x', shape))
    _lib.TIMING = []
    try:
        y, dx, grads = _run_layer(m, x)
        names = {t[0] for t in _lib.TIMING}
    finally:
        _lib.TIMING = None
    assert not any('im2col' in n or 'col2im' in n for n in names), names
    sdr = round_conv_weights(sd)
    xr = x.clone().requires_grad_(True)
    w = sdr['conv3d.weight'].clone().requires_grad_(True)
    yo = O.causal_conv3d(xr, w, sdr['conv3d.bias'], stride=stride)
    assert_close(y, yo, 1e-3, 1e-5 * yo.abs().max().item(), 'narrow fwd')
    yo.backward(bf16_round((2.0 / yo.numel()) * y))
    assert dx.shape == xr.grad.shape
    assert_close(dx, xr.grad, BF16_ULP, BF16_ULP * xr.grad.abs().max().item(), 'narrow dgrad')
    assert grads['conv3d.weight'].shape == w.grad.shape
    assert_close(grads['conv3d.weight'], w.grad, 2e-3, 1e-3 * w.grad.abs().max().item(), 'narrow wgrad')
    # the optimizer refreshes the channel-padded bf16 operand in place
    from open_genie_b200.optim import FusedAdamW
    opt = FusedAdamW(m.parameters(), lr=0.05)
    opt.step()
    packed = m.conv3d.packed().float().view(cout, 27, 64)
    wnow = m.conv3d.weight.detach().permute(0, 2, 3, 4, 1).reshape(cout, 27, cin)
    assert torch.equal(packed[:, :, :cin], wnow.to(torch.bfloat16).float()) and float(packed[:, :, cin:].abs().max()) == 0.0


def test_spacetime_downsample_im2col_path(golden, monkeypatch):
    monkeypatch.setenv('OG_STRIDED_IM2COL', '1')        # the explicit path stays available for Cin not in 64Z
    from open_genie_b200.module.video import SpaceTimeDownsample
    g = golden('layers.pt')['spacetime_downsample']
    m = SpaceTimeDownsample(64, 3, 64, time_factor=2, space_factor=2)
    sd = det_weights(m)
    m.to(DEV)
    m.go_down.out_f32 = True
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    y, dx, grads = _run_layer(m, x)
    assert y.shape == (2, 64, 2, 4, 4)
    sdr = round_conv_weights(sd)
    xr = x.clone().requires_grad_(True)
    w = sdr['go_down.conv3d.weight'].clone().requires_grad_(True)
    yo = O.causal_conv3d(xr, w, sdr['go_down.conv3d.bias'], stride=(2, 2, 2))
    assert_close(y, yo, 1e-3, 1e-5 * yo.abs().max().item(), 'strided conv fwd')
    assert rel_l2(at_sample(y, 'layers.spacetime_downsample.y', g['y']), g['y']) < 1e-2
    yo.backward(bf16_round((2.0 / yo.numel()) * y))
    # dcol is stored in bf16 before col2im sums up to 27 of them
    assert rel_l2(dx, xr.grad) < 1e-2
    assert_close(grads['go_down.conv3d.weight'], w.grad, 2e-3, 1e-3 * w.grad.abs().max().item(), 'strided wgrad')


def test_video_residual_block(golden):
    from open_genie_b200.module.video import VideoResidualBlock
    g = golden('layers.pt')['video_residual']
    m = VideoResidualBlock(64, 128)
    sd = det_weights(m)
    m.to(DEV)
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    y, dx, grads = _run_layer(m, x)
    # oracle composed with the product's rounding points (bf16 between kernels)
    import torch.nn.functional as F
    sdr = round_conv_weights(sd)
    h = bf16_round(F.silu(F.group_norm(x, 1, sdr['main.0.weight'], sdr['main.0.bias'])))
    h = bf16_round(F.conv3d(h, sdr['main.2.weight'], sdr['main.2.bias'], padding=1))
    h = bf16_round(F.silu(F.group_norm(h, 1, sdr['main.4.weight'], sdr['main.4.bias'])))
    yo = F.conv3d(h, sdr['main.6.weight'], sdr['main.6.bias'], padding=1) + F.conv3d(x, sdr['res.1.weight'],
                                                                                    sdr['res.1.bias'])
    assert_close(y, bf16_round(yo), 2 * BF16_ULP, 2 * BF16_ULP * yo.abs().max().item(), 'residual block fwd')
    assert rel_l2(at_sample(y, 'layers.video_residual.y', g['y']), g['y']) < 2e-2    # vs the unrounded reference run
    assert rel_l2(at_sample(dx, 'layers.video_residual.dx', g['dx']), g['dx']) < 5e-2
    for k, v in g['grads']['full'].items():
        assert rel_l2(grads[k], v) < 5e-2, k
    for k, n in g['grads']['norm'].items():
        assert abs(grads[k].norm().item() - n) / n < 5e-2, k


def test_blur_pool_and_downsampling_residual_block(golden):
    from open_genie_b200 import ops
    from open_genie_b200.module.video import BlurPooling3d, VideoResidualBlock
    k = golden('kats.pt')
    xb = bf16_round(O.det_uniform('kat.blur.x', (1, 8, 4, 8, 8)))
    bp = BlurPooling3d(8, 3).to(DEV)
    assert torch.equal(bp.blur.cpu(), k['blur3'])
    xg = xb.to(DEV).requires_grad_(True)
    y = bp(xg)
    xr = xb.clone().requires_grad_(True)
    yo = O.blur_pool3d(xr, 3, 2, 2)
    gy = bf16_round(O.det_uniform('blur.gy', tuple(yo.shape)))
    y.backward(gy.to(DEV).to(y.dtype))
    yo.backward(gy)
    assert_close(ops.to_reference(y), bf16_round(yo), BF16_ULP, BF16_ULP * yo.abs().max().item(), 'blur fwd')
    assert_close(xg.grad, xr.grad, 2 * BF16_ULP, 2 * BF16_ULP * xr.grad.abs().max().item(), 'blur bwd')
    g = golden('layers.pt')['video_residual_down']
    m = VideoResidualBlock(64, 128, downsample=(2, 2))
    det_weights(m)
    m.to(DEV)
    assert {'res.0.blur', 'main.3.blur'} <= set(m.state_dict())
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    y, dx, grads = _run_layer(m, x)
    assert y.shape == (2, 128, 2, 4, 4)
    assert rel_l2(at_sample(y, 'layers.video_residual_down.y', g['y']), g['y']) < 2e-2
    assert rel_l2(at_sample(dx, 'layers.video_residual_down.dx', g['dx']), g['dx']) < 6e-2
    for key, n in g['grads']['norm'].items():
        assert abs(grads[key].norm().item() - n) / n < 6e-2, key


def test_depth2spacetime_upsample(golden):
    from open_genie_b200.module.video import DepthToSpaceTimeUpsample
    g = golden('layers.pt')['depth2spacetime_upsample']
    m = DepthToSpaceTimeUpsample(64, kernel_size=3, time_factor=2, space_factor=2)
    sd = det_weights(m)
    m.to(DEV)
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    y, dx, grads = _run_layer(m, x)
    assert y.shape == (2, 64, 8, 16, 16)
    yo = O.depth2spacetime_upsample(round_conv_weights(sd), '', x, 2, 2)
    assert_close(y, bf16_round(yo), BF16_ULP, BF16_ULP * yo.abs().max().item(), 'upsample fwd')
    assert rel_l2(at_sample(dx, 'layers.depth2spacetime_upsample.dx', g['dx']), g['dx']) < 3e-2
    assert rel_l2(grads['go_up.0.conv3d.weight'].norm(), torch.tensor(g['grads']['norm']['go_up.0.conv3d.weight'])) < 3e-2


def test_adaptive_group_norm(golden):
    from open_genie_b200.module.norm import AdaptiveGroupNorm
    g = golden('layers.pt')['adaptive_group_norm']
    m = AdaptiveGroupNorm(6, 8, 64)
    det_weights(m)
    m.to(DEV)
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    cond = O.det_uniform('layers.cond', (2, 6, 2, 4, 4)).sign().to(DEV)
    y, dx, grads = _run_layer(m, x, cond)
    assert y.shape == (2, 64, 4, 8, 8)
    assert_close(at_sample(y, 'layers.adaptive_group_norm.y', g['y']), bf16_round(g['y']), BF16_ULP,
                 BF16_ULP * g['y'].abs().max().item(), 'AdaGN fwd')
    assert rel_l2(at_sample(dx, 'layers.adaptive_group_norm.dx', g['dx']), g['dx']) < 2e-2
    for k, v in g['grads']['full'].items():
        assert rel_l2(grads[k], v) < 2e-2, k


@pytest.mark.parametrize('groups,act', [(1, 'silu'), (8, 'none'), (8, 'silu')])
def test_group_norm_act(groups, act):
    import torch.nn.functional as F
    from open_genie_b200 import ops
    x = bf16_round(O.det_uniform(f'gn.x.{groups}', (2, 128, 4, 16, 16)) * 2 + 0.3)
    gamma = (1 + O.det_uniform('gn.g', (128,), 0.2)).to(DEV).requires_grad_(True)
    beta = O.det_uniform('gn.b', (128,), 0.2).to(DEV).requires_grad_(True)
    xg = x.to(DEV).requires_grad_(True)
    y = ops.group_norm_act(xg, gamma, beta, groups, 1e-5, act)
    gy = bf16_round(O.det_uniform('gn.gy', tuple(y.shape)))
    y.backward(gy.to(DEV).to(y.dtype))
    xr = x.clone().requires_grad_(True)
    gr = gamma.detach().cpu().requires_grad_(True)
    br = beta.detach().cpu().requires_grad_(True)
    yo = F.group_norm(xr, groups, gr, br, 1e-5)
    yo = F.silu(yo) if act == 'silu' else yo
    yo.backward(gy)
    assert_close(ops.to_reference(y), bf16_round(yo), BF16_ULP, BF16_ULP, 'GN fwd')
    assert_close(xg.grad, xr.grad, 2 * BF16_ULP, 2 * BF16_ULP * xr.grad.abs().max().item(), 'GN dx')
    assert_close(gamma.grad, gr.grad, 2e-3, 2e-3 * gr.grad.abs().max().item(), 'GN dgamma')
    assert_close(beta.grad, br.grad, 2e-3, 2e-3 * br.grad.abs().max().item(), 'GN dbeta')


def test_pixel_shuffle_roundtrip_and_values():
    from open_genie_b200 import ops
    x = bf16_round(O.det_uniform('ps.x', (2, 64 * 8, 2, 4, 4)))
    y = ops.pixel_shuffle3d(x.to(DEV), 2, 2, 2)
    b, cc, t, h, w = x.shape
    ref = x.reshape(b, 64, 2, 2, 2, t, h, w).permute(0, 1, 5, 2, 6, 3, 7, 4).reshape(b, 64, t * 2, h * 2, w * 2)
    assert torch.equal(ops.to_reference(y).cpu(), ref)          # pure data movement: bit exact
    from open_genie_b200 import _lib
    back = ops.empty_internal(b, cc, t, h, w)
    _lib.call('og_pixel_shuffle3d', back.data_ptr(), y.data_ptr(), 1, b, t, h, w, 64, 2, 2, 2,
              torch.cuda.current_stream().cuda_stream)
    assert torch.equal(ops.to_reference(back).cpu(), x)


@pytest.mark.parametrize('d', [8, 10, 18])
def test_lfq_matches_golden(golden, d):
    from open_genie_b200.module.quantization import LookupFreeQuantization
    g = golden('lfq.pt')[f'd{d}']
    n = g['n']
    m = LookupFreeQuantization(d, input_dim=d).to(DEV).train()
    x = O.det_uniform(f'lfq.x.{d}', (2, n // 2, d), 0.6).to(DEV).requires_grad_(True)
    (q, idx), loss = m(x)
    gq = O.det_uniform(f'lfq.gq.{d}', tuple(q.shape)).to(DEV)
    (loss + (q * gq).sum()).backward()
    assert torch.equal(idx.cpu(), g['idxs'])                    # indices: bit exact
    assert torch.equal(q.detach().cpu(), g['out'])              # STE value x + (sign(x) - x): bit exact
    assert_close(loss, g['loss'], 1e-3, 1e-5, 'lfq loss')
    assert_close(x.grad, g['dx'], 1e-3, 1e-5 * g['dx'].abs().max().item() + 1e-6, 'lfq dx')
    m.eval()
    (q2, idx2), l2 = m(x.detach())
    assert l2 is None and torch.equal(idx2.cpu(), g['idxs']) and torch.equal(q2.cpu(), x.detach().sign().cpu())


def test_lfq_kats(golden):
    from open_genie_b200.module.quantization import LookupFreeQuantization
    k = golden('kats.pt')
    m = LookupFreeQuantization(4, input_dim=4).to(DEV).eval()
    (q, idx), _ = m(k['lfq4_x'].to(DEV))
    assert torch.equal(q.cpu(), k['lfq4_quant']) and torch.equal(idx.cpu(), k['lfq4_idx'])
    assert torch.equal(m.bit_mask.cpu(), k['bit_mask'])


def test_lfq_flat_distribution_edge_case():
    """x ~ 0 makes every one of the 2^D codes exceed the clamp eps: exercises the no-row-skipped path."""
    from open_genie_b200.module.quantization import LookupFreeQuantization
    d = 12
    x = (O.det_uniform('lfq.flat', (1, 16, d)) * 2e-4).requires_grad_(True)
    (_, _), lo = O.lfq(x, d, True)
    lo.backward()
    m = LookupFreeQuantization(d, input_dim=d).to(DEV).train()
    xg = x.detach().to(DEV).requires_grad_(True)
    (_, _), l = m(xg)
    l.backward()
    assert_close(l, lo, 1e-3, 1e-5, 'lfq loss (flat)')
    assert_close(xg.grad, x.grad, 2e-3, 2e-3 * x.grad.abs().max().item(), 'lfq dx (flat)')


def test_mse_loss_and_layout_roundtrip():
    from open_genie_b200 import ops
    v = O.det_uniform('mse.v', (2, 3, 4, 16, 16))
    r = O.det_uniform('mse.r', (2, 3, 4, 16, 16))
    ri = ops.to_internal(r.to(DEV), torch.float32).requires_grad_(True)
    loss = ops.mse_loss(ri, v.to(DEV))
    loss.backward()
    ref = torch.nn.functional.mse_loss(r, v)
    assert_close(loss, ref, 1e-5, 1e-7, 'mse')
    gref = 2 * (r - v) / r.numel()
    assert_close(ops.to_reference(ri.grad.float()), gref, BF16_ULP, 1e-9, 'mse grad')
    # layout round trip is exact for bf16-representable data
    x = bf16_round(O.det_uniform('rt.x', (2, 18, 4, 8, 8)))
    assert torch.equal(ops.to_reference(ops.to_internal(x.to(DEV))).cpu(), x)


def test_operand_swapped_gemm_matches_plain_tiles(monkeypatch):
    """Cout = 128 layers with >= 2 x #SM voxel tiles run the operand-swapped GEMM (D^T = W . X^T, transposing
    epilogue). At the full tokenizer size (8 x 16 x 64 x 64, C = 128) its output, fused GroupNorm statistics and
    data gradient must equal those of the plain 128 x 128 tile path (OG_IGEMM_SWAP=0): same k order, same fp32
    accumulation, so bit-exact bf16 — and a small corner is checked against the fp32 oracle."""
    import torch.nn.functional as F
    from open_genie_b200.module.video import CausalConv3d
    from open_genie_b200 import ops
    torch.manual_seed(0)
    m = CausalConv3d(128, 128, 3).to(DEV)
    x = torch.randn(8, 128, 16, 64, 64, device=DEV)
    xi = ops.to_internal(x, torch.bfloat16)

    def run():
        xin = xi.detach().clone().requires_grad_(True)
        y = m(xin)
        g = torch.sin(torch.arange(y.numel(), device=DEV, dtype=torch.float32)).view_as(y).to(y.dtype)
        y.backward(g)
        return y.detach().float(), xin.grad.detach().float()

    y1, dx1 = run()
    monkeypatch.setenv('OG_IGEMM_SWAP', '0')
    y0, dx0 = run()
    assert torch.equal(y1, y0), (y1 - y0).abs().max().item()
    assert torch.equal(dx1, dx0), (dx1 - dx0).abs().max().item()
    # corner of sample 0 against the oracle (causal front pad in time, symmetric in space)
    w = bf16_round(m.conv3d.weight.detach().float().cpu())
    b = m.conv3d.bias.detach().float().cpu()
    xc = bf16_round(ops.to_reference(xi[:1, :, :4, :10, :10].float()).cpu())
    yo = O.causal_conv3d(xc, w, b)[:, :, :, :8, :8]
    got = ops.to_reference(y1[:1, :, :4, :8, :8]).cpu()
    assert_close(got, bf16_round(yo), BF16_ULP, BF16_ULP * yo.abs().max().item(), 'swapped GEMM corner vs oracle')


def test_zero_arena_gradients_match_plain_allocation():
    """A residual block run with the step-scoped zero arena (gradient accumulators, GroupNorm sums and
    reduction buffers carved from one buffer, one fill per step) gives the same output and gradients as with
    per-tensor torch.zeros — over three simulated steps (first measures, second allocates, third recycles).
    The block has no ill-conditioned stage, so the only run-to-run noise is the order of fp32 atomics."""
    from open_genie_b200 import ops
    from open_genie_b200.module.video import VideoResidualBlock
    m = VideoResidualBlock(64, 128)
    det_weights(m)
    m.to(DEV)
    x = bf16_round(O.det_uniform('layers.x', (2, 64, 4, 8, 8)))
    dev = None
    try:
        ops.enable_zero_arena(False)
        y0, dx0, g0 = _run_layer(m, x)
        ops.enable_zero_arena(True)
        for it in range(3):
            m.zero_grad(set_to_none=True)          # the arena contract: gradients are released every step
            ops.mark_step()
            y1, dx1, g1 = _run_layer(m, x)
            assert_close(y1, y0, BF16_ULP, BF16_ULP * y0.abs().max().item(), f'arena fwd (step {it})')
            assert_close(dx1, dx0, 2 * BF16_ULP, 2 * BF16_ULP * dx0.abs().max().item(), f'arena dx (step {it})')
            for k in g0:
                assert_close(g1[k], g0[k], 2e-3, 2e-3 * g0[k].abs().max().item(), f'arena grad {k} (step {it})')
        assert ops.ZERO_ARENA.bytes_in_use() > 0                           # the arena was really used
    finally:
        ops.enable_zero_arena(False)
