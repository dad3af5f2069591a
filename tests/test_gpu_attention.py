"""GPU parity: RoPE+LayerNorm, tcgen05 flash attention, temporal attention, SpaceTimeAttention block."""
import pytest
import torch
import torch.nn.functional as F

from helpers import assert_close, at_sample, bf16_round, det_weights, rel_l2
from oracle import fixtures as fx
from oracle import genie_oracle as O

pytestmark = pytest.mark.gpu
DEV = 'cuda'
BF16_ULP = 2.0 ** -7


def _call(name, *a):
    from open_genie_b200 import _lib
    _lib.call(name, *a, torch.cuda.current_stream().cuda_stream)


@pytest.mark.parametrize('kind,C', [('2d', 128), ('1d', 512), ('2d', 256)])
def test_rope_layernorm_fwd_bwd(kind, C):
    B, T, H, W = 2, 4, 8, 8
    x = bf16_round(O.det_uniform(f'rl.x.{kind}', (B, T, H, W, C)))
    freq = O.rope_freq(C, kind)
    gamma = 1 + O.det_uniform('rl.g', (C,), 0.2)
    beta = O.det_uniform('rl.b', (C,), 0.2)
    gy = bf16_round(O.det_uniform('rl.gy', (B, T, H, W, C)))
    # oracle: spatial -> sequences are frames; temporal -> sequences are pixels
    xr = x.clone().requires_grad_(True)
    gr, br = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    if kind == '2d':
        seq = xr.reshape(B * T, H * W, C)
        yo = F.layer_norm(O.rope(seq, freq), (C,), gr, br).reshape(B, T, H, W, C)
        pos_div, pos_mod = 1, H * W
    else:
        seq = xr.permute(0, 2, 3, 1, 4).reshape(B * H * W, T, C)
        yo = F.layer_norm(O.rope(seq, freq), (C,), gr, br).reshape(B, H, W, T, C).permute(0, 3, 1, 2, 4)
        pos_div, pos_mod = H * W, T
    yo.backward(gy)
    xd = x.to(DEV).to(torch.bfloat16).contiguous()
    y = torch.empty_like(xd)
    fq, ga, be = freq.to(DEV), gamma.to(DEV), beta.to(DEV)
    rows = B * T * H * W
    _call('og_rope_ln_fwd', xd.data_ptr(), fq.data_ptr(), ga.data_ptr(), be.data_ptr(), 1e-5, y.data_ptr(), rows, C,
          pos_div, pos_mod, None)
    assert_close(y.float(), bf16_round(yo), BF16_ULP, BF16_ULP, 'rope+ln fwd')
    # the precomputed (cos, sin) table holds the same sincosf values: bit-identical output, forward and backward
    tab = torch.empty((pos_mod, C // 2, 2), device=DEV)
    _call('og_rope_table', fq.data_ptr(), pos_mod, C, tab.data_ptr())
    y_t = torch.empty_like(xd)
    _call('og_rope_ln_fwd', xd.data_ptr(), fq.data_ptr(), ga.data_ptr(), be.data_ptr(), 1e-5, y_t.data_ptr(), rows, C,
          pos_div, pos_mod, tab.data_ptr())
    assert torch.equal(y_t, y), 'table and sincosf paths differ (forward)' 
    g = gy.to(DEV).to(torch.bfloat16).contiguous()
    dx = torch.empty_like(xd)
    dg, db = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
    _call('og_rope_ln_bwd', xd.data_ptr(), fq.data_ptr(), ga.data_ptr(), 1e-5, g.data_ptr(), None, None, None,
          dx.data_ptr(), dg.data_ptr(), db.data_ptr(), rows, C, pos_div, pos_mod, None)
    dx_t = torch.empty_like(xd)
    dg_t, db_t = torch.zeros(C, device=DEV), torch.zeros(C, device=DEV)
    _call('og_rope_ln_bwd', xd.data_ptr(), fq.data_ptr(), ga.data_ptr(), 1e-5, g.data_ptr(), None, None, None,
          dx_t.data_ptr(), dg_t.data_ptr(), db_t.data_ptr(), rows, C, pos_div, pos_mod, tab.data_ptr())
    assert torch.equal(dx_t, dx), 'table and sincosf paths differ (backward)' 
    assert_close(dx.float(), xr.grad, 2 * BF16_ULP, 2 * BF16_ULP * xr.grad.abs().max().item(), 'rope+ln dx')
    assert_close(dg, gr.grad, 2e-3, 2e-3 * gr.grad.abs().max().item(), 'dgamma')
    assert_close(db, br.grad, 2e-3, 2e-3 * br.grad.abs().max().item(), 'dbeta')


# amp = 2 with 8 heads (scale = 1.0) gives scores of +-100: the running row maximum jumps by far more than the
# lazy-rescale threshold (2^8) between key tiles, so the in-TMEM rescale of O is exercised, not only the first tile
@pytest.mark.parametrize('S,nh,amp', [(64, 2, 0.5), (256, 2, 0.5), (320, 1, 0.5), (1024, 4, 0.5), (640, 8, 2.0)])
def test_flash_attention_fwd_bwd(S, nh, amp):
    nseq, C = 3, 64 * nh
    scale = nh * 64 ** -0.5                                   # the reference's (quirky) scale, attention.py:195
    q = bf16_round(O.det_uniform(f'fa.q.{S}', (nseq, S, C), amp))
    k = bf16_round(O.det_uniform(f'fa.k.{S}', (nseq, S, C), amp))
    v = bf16_round(O.det_uniform(f'fa.v.{S}', (nseq, S, C)))
    do = bf16_round(O.det_uniform(f'fa.do.{S}', (nseq, S, C)))
    qr, kr, vr = (t.clone().requires_grad_(True) for t in (q, k, v))
    sp = lambda t: t.reshape(nseq, S, nh, 64).transpose(1, 2)
    oo = F.scaled_dot_product_attention(sp(qr), sp(kr), sp(vr), scale=scale).transpose(1, 2).reshape(nseq, S, C)
    oo.backward(do)
    dev = lambda t: t.to(DEV).to(torch.bfloat16).contiguous()
    qd, kd, vd, dod = dev(q), dev(k), dev(v), dev(do)
    out = torch.empty_like(qd)
    lse = torch.empty((nseq, nh, S), device=DEV)
    _call('og_flash_attn_fwd', qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), out.data_ptr(), None, None, lse.data_ptr(),
          nseq, S, C, nh, scale)
    # P is rounded to bf16 before the PV product: tolerance of one bf16 ulp of the output scale
    assert_close(out.float(), oo, 2 * BF16_ULP, 2 * BF16_ULP * oo.abs().max().item(), 'flash fwd')
    lse_ref = torch.logsumexp(torch.einsum('bhqd,bhkd->bhqk', sp(q), sp(k)) * scale, -1)
    assert_close(lse, lse_ref, 1e-3, 1e-3, 'lse')
    dq, dk, dv = torch.empty_like(qd), torch.empty_like(qd), torch.empty_like(qd)
    delta = torch.empty_like(lse)
    _call('og_flash_attn_bwd', qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), out.data_ptr(), dod.data_ptr(),
          lse.data_ptr(), delta.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), nseq, S, C, nh, scale)
    for name, got, ref in (('dq', dq, qr.grad), ('dk', dk, kr.grad), ('dv', dv, vr.grad)):
        assert rel_l2(got.float().cpu(), ref) < 2e-2, (name, rel_l2(got.float().cpu(), ref))


# Many more work items than SMs with ODD tile counts per item (1, 3, 5): every persistent CTA walks several items, so the
# running-counter barrier parities of og_flash_attn_fwd2 / bwd3 cross item boundaries on both phases of every barrier.
# Reference: torch's SDPA in fp32 on the GPU (the small cases above pin the kernels to the CPU oracle values).
@pytest.mark.parametrize('S,nseq,nh', [(64, 200, 2), (320, 120, 1), (640, 40, 2)])
def test_flash_attention_many_items_per_cta(S, nseq, nh):
    C = 64 * nh
    scale = nh * 64 ** -0.5
    g = torch.Generator(device='cpu').manual_seed(S)
    q, k, v, do = (torch.randn(nseq, S, C, generator=g).mul_(0.5).to(DEV).to(torch.bfloat16) for _ in range(4))
    sp = lambda t: t.float().reshape(nseq, S, nh, 64).transpose(1, 2)
    qr, kr, vr = (t.clone().requires_grad_(True) for t in (q, k, v))
    oo = F.scaled_dot_product_attention(sp(qr), sp(kr), sp(vr), scale=scale).transpose(1, 2).reshape(nseq, S, C)
    oo.backward(do.float())
    out = torch.empty_like(q)
    lse = torch.empty((nseq, nh, S), device=DEV)
    _call('og_flash_attn_fwd', q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), None, None, lse.data_ptr(),
          nseq, S, C, nh, scale)
    assert rel_l2(out.float().cpu(), oo.detach().cpu()) < 1e-2
    dq, dk, dv = torch.empty_like(q), torch.empty_like(q), torch.empty_like(q)
    delta = torch.empty_like(lse)
    _call('og_flash_attn_bwd', q.data_ptr(), k.data_ptr(), v.data_ptr(), out.data_ptr(), do.data_ptr(), lse.data_ptr(),
          delta.data_ptr(), dq.data_ptr(), dk.data_ptr(), dv.data_ptr(), nseq, S, C, nh, scale)
    for name, got, ref in (('dq', dq, qr.grad), ('dk', dk, kr.grad), ('dv', dv, vr.grad)):
        assert rel_l2(got.float().cpu(), ref.float().cpu()) < 2e-2, (name, rel_l2(got.float().cpu(), ref.float().cpu()))


@pytest.mark.parametrize('bcast', [False, True])
def test_temporal_attention_fwd_bwd(bcast):
    B, T, P, nh = 2, 8, 24, 2
    C = 64 * nh
    scale = nh * 64 ** -0.5
    q = bf16_round(O.det_uniform('ta.q', (B, T, P, C), 0.5))
    do = bf16_round(O.det_uniform('ta.do', (B, T, P, C)))
    if bcast:
        k = bf16_round(O.det_uniform('ta.k', (B, T, C), 0.5))
        v = bf16_round(O.det_uniform('ta.v', (B, T, C)))
    else:
        k, v = q, q
    qr = q.clone().requires_grad_(True)
    kr = k.clone().requires_grad_(True) if bcast else qr
    vr = v.clone().requires_grad_(True) if bcast else qr
    sq = lambda t: t.permute(0, 2, 1, 3).reshape(B * P, T, nh, 64).transpose(1, 2)
    if bcast:
        ex = lambda t: t[:, None].expand(B, P, T, C).reshape(B * P, T, nh, 64).transpose(1, 2)
        oo = F.scaled_dot_product_attention(sq(qr), ex(kr), ex(vr), is_causal=True, scale=scale)
    else:
        oo = F.scaled_dot_product_attention(sq(qr), sq(qr), sq(qr), is_causal=True, scale=scale)
    oo = oo.transpose(1, 2).reshape(B, P, T, C).permute(0, 2, 1, 3)
    oo.backward(do)
    dev = lambda t: t.to(DEV).to(torch.bfloat16).contiguous()
    qd, kd, vd, dod = dev(q), dev(k), dev(v), dev(do)
    out = torch.empty_like(qd)
    _call('og_temporal_attn_fwd', qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), None, out.data_ptr(), B, T, P, C, nh,
          scale, int(bcast))
    assert_close(out.float(), bf16_round(oo), 2 * BF16_ULP, 2 * BF16_ULP * oo.abs().max().item(), 'temporal fwd')
    dq = torch.empty_like(qd)
    if bcast:
        dkb, dvb = torch.zeros((B, T, C), device=DEV), torch.zeros((B, T, C), device=DEV)
        _call('og_temporal_attn_bwd', qd.data_ptr(), kd.data_ptr(), vd.data_ptr(), dod.data_ptr(), dq.data_ptr(), None,
              None, dkb.data_ptr(), dvb.data_ptr(), B, T, P, C, nh, scale, 1)
        assert rel_l2(dq.float().cpu(), qr.grad) < 1e-2
        assert rel_l2(dkb.cpu(), kr.grad) < 1e-2 and rel_l2(dvb.cpu(), vr.grad) < 1e-2
    else:
        dk, dv = torch.empty_like(qd), torch.empty_like(qd)
        _call('og_temporal_attn_bwd', qd.data_ptr(), qd.data_ptr(), qd.data_ptr(), dod.data_ptr(), dq.data_ptr(),
              dk.data_ptr(), dv.data_ptr(), None, None, B, T, P, C, nh, scale, 0)
        tot = dq.float() + dk.float() + dv.float()
        assert rel_l2(tot.cpu(), qr.grad) < 1e-2


@pytest.mark.parametrize('case', range(4))
def test_spacetime_attention_block_against_reference_golden(golden, case):
    from open_genie_b200.module.attention import SpaceTimeAttention
    transpose, cond_dim, shape = fx.ST_BLOCK_CASES[case]
    tag = f't{int(transpose)}_c{cond_dim or 0}'
    g = golden('st_block.pt')[tag]
    kw = {'time_attn_kw': {'key_dim': cond_dim}} if cond_dim else {}
    m = SpaceTimeAttention(n_head=2, d_head=64, transpose=transpose, **kw)
    det_weights(m)
    m.to(DEV)
    x = O.det_uniform(f'st.x.{tag}', shape).to(DEV).requires_grad_(True)
    t = shape[2] if transpose else shape[1]
    cond = O.det_uniform('st.cond', (2, t, 4)).sign().to(DEV) if cond_dim else None
    y = m(x, cond=(None, cond)) if cond_dim else m(x)
    assert tuple(y.shape) == tuple(shape)
    gy = (2.0 / y.numel()) * y.detach().float()
    y.backward(gy.to(y.dtype))
    assert rel_l2(at_sample(y, f'st_block.{tag}.y', g['y']), g['y']) < 2e-2
    assert rel_l2(at_sample(x.grad, f'st_block.{tag}.dx', g['dx']), g['dx']) < 6e-2
    grads = {k: p.grad.float().cpu() for k, p in m.named_parameters() if p.grad is not None}
    assert set(grads) == set(g['grads']['norm'])
    for k, v in g['grads']['full'].items():
        assert rel_l2(grads[k], v) < 8e-2, (k, rel_l2(grads[k], v))
    for k, n in g['grads']['norm'].items():
        assert abs(grads[k].norm().item() - n) / n < 8e-2, k
