"""CPU: the oracle (oracle/genie_oracle.py) against the golden vectors produced by the REAL reference
(oracle/make_golden.py, run in the build container where /root/reference exists). This is what pins the
oracle; the GPU tests then compare the CUDA path with the oracle and with the same vectors."""
import torch

import open_genie_b200 as og
from oracle import fixtures as fx
from oracle import genie_oracle as O


def _sd_for(module):
    shapes = {k: tuple(v.shape) for k, v in module.state_dict().items()}
    sd = O.det_state_dict(shapes)
    full = {k: v.detach().clone() for k, v in module.state_dict().items()}
    full.update(sd)
    return full


def _close(a, b, rtol=1e-4, atol=1e-5):
    assert torch.allclose(torch.as_tensor(a).float(), torch.as_tensor(b).float(), rtol=rtol, atol=atol), \
        (torch.as_tensor(a).float() - torch.as_tensor(b).float()).abs().max()


def test_kats(golden):
    k = golden('kats.pt')
    for which, ref in k['schedule'].items():
        assert torch.equal(O.maskgit_schedule(10, (16, 16), which), ref)
    assert k['schedule']['linear'].tolist() == [1, 6, 11, 17, 23, 28, 34, 40, 46, 50]      # SURVEY.md §8c
    (q, idx), loss = O.lfq(k['lfq4_x'], 4, training=False)
    assert loss is None and torch.equal(q, k['lfq4_quant']) and torch.equal(idx, k['lfq4_idx'])
    assert idx.flatten().tolist() == [9, 0, 15] and k['bit_mask'].tolist() == [8, 4, 2, 1]
    assert torch.equal(O.lfq_bit_mask(4), k['bit_mask'])
    _close(O.rope_freq(8, '1d'), k['rope_1d_c8'])
    _close(O.rope_freq(8, '2d'), k['rope_2d_c8'])
    _close(O.blur_kernel(3), k['blur3'])
    _close(O.blur_pool3d(O.det_uniform('kat.blur.x', (1, 4, 4, 8, 8)), 3, 2, 2), k['blur_pool_out'])


def test_lfq_training_vectors(golden):
    g = golden('lfq.pt')
    for d in (8, 10, 18):
        e = g[f'd{d}']
        x = O.det_uniform(f'lfq.x.{d}', (2, e['n'] // 2, d), 0.6).requires_grad_(True)
        (q, idx), loss = O.lfq(x, d, training=True)
        (loss + (q * O.det_uniform(f'lfq.gq.{d}', tuple(q.shape))).sum()).backward()
        assert torch.equal(idx, e['idxs']) and torch.equal(q.detach(), e['out'])
        _close(loss, e['loss'])
        _close(x.grad, e['dx'], 1e-4, 1e-6)


def test_layer_vectors(golden):
    from open_genie_b200.module.norm import AdaptiveGroupNorm
    from open_genie_b200.module.video import (CausalConv3d, DepthToSpaceTimeUpsample, SpaceTimeDownsample,
                                              VideoResidualBlock)
    g = golden('layers.pt')

    def y_of(name, y):            # the golden stores each output on a deterministic sample of its values
        return O.det_sample(y, f'layers.{name}.y', g[name]['y'].numel())
    x = O.det_uniform('layers.x', (2, 64, 4, 8, 8))
    sd = _sd_for(CausalConv3d(64, 64, 3))
    _close(y_of('causal_conv3d', O.causal_conv3d(x, sd['conv3d.weight'], sd['conv3d.bias'])), g['causal_conv3d']['y'])
    sd = _sd_for(SpaceTimeDownsample(64, 3, 64, time_factor=2, space_factor=2))
    _close(y_of('spacetime_downsample', O.spacetime_downsample(sd, '', x, 2, 2)), g['spacetime_downsample']['y'])
    sd = _sd_for(VideoResidualBlock(64, 128))
    _close(y_of('video_residual', O.video_residual_block(sd, '', x)), g['video_residual']['y'])
    sd = _sd_for(VideoResidualBlock(64, 128, downsample=(2, 2)))
    _close(y_of('video_residual_down', O.video_residual_block(sd, '', x, downsample=(2, 2))), g['video_residual_down']['y'])
    sd = _sd_for(DepthToSpaceTimeUpsample(64, kernel_size=3, time_factor=2, space_factor=2))
    _close(y_of('depth2spacetime_upsample', O.depth2spacetime_upsample(sd, '', x, 2, 2)), g['depth2spacetime_upsample']['y'])
    sd = _sd_for(AdaptiveGroupNorm(6, 8, 64))
    cond = O.det_uniform('layers.cond', (2, 6, 2, 4, 4)).sign()
    _close(y_of('adaptive_group_norm', O.adaptive_group_norm(sd, '', x, cond, 8)), g['adaptive_group_norm']['y'])


def test_tokenizer_vectors(golden):
    g = golden('tokenizer_mini.pt')
    tok = og.VideoTokenizer(fx.MINI_ENC, fx.MINI_DEC, d_codebook=fx.MINI_D_CODEBOOK, gan_loss_weight=0,
                            perc_loss_weight=0)
    assert sum(p.numel() for p in tok.parameters()) == g['n_params']
    sd = {k: v.requires_grad_(v.dtype.is_floating_point) for k, v in _sd_for(tok).items()}
    video = O.det_uniform('tokenizer.video', fx.MINI_VIDEO_SHAPE)
    q, idx = O.tokenizer_tokenize(sd, fx.MINI_ENC, video, fx.MINI_D_CODEBOOK)
    assert torch.equal(idx, g['idxs']) and torch.equal(q.detach(), g['quant'])
    _close(O.tokenizer_decode(sd, fx.MINI_DEC, g['quant']), g['decode'], 2e-4, 2e-5)
    loss, (rec, ql), rec_video, _ = O.tokenizer_forward(sd, fx.MINI_ENC, fx.MINI_DEC, video, fx.MINI_D_CODEBOOK)
    _close(loss, g['loss']); _close(rec, g['rec_loss']); _close(ql, g['quant_loss'])
    _close(rec_video, g['rec_video'], 2e-4, 2e-5)
    loss.backward()
    for k, n in g['grads']['norm'].items():
        assert abs(sd[k].grad.norm().item() - n) <= 2e-3 * n + 1e-7, k
    for k, v in g['grads']['full'].items():
        if k.startswith('dec_layers'):
            _close(sd[k].grad, v, 2e-3, 1e-6 + 2e-3 * v.abs().max().item())
