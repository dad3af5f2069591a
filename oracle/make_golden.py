"""oracle/make_golden.py — generate tests/golden/*.pt by RUNNING THE REAL REFERENCE.   TEST INFRASTRUCTURE.

Run in the build container only (needs /root/reference, which does not exist on the GPU box):

    python oracle/make_golden.py            # writes tests/golden/*.pt, asserts oracle == reference

The reference modules are imported unmodified (a `lightning` shim is put on sys.path because that
package is not installed here), instantiated in their HEAD-valid configurations (SURVEY.md §8),
loaded with RNG-free deterministic weights (oracle.genie_oracle.det_state_dict) and run on CPU fp32.
What is stored is small: configuration, outputs, losses and gradients — weights and inputs are
re-derived from their closed form by the tests.  While generating, every output is also compared
with the restatement in oracle/genie_oracle.py; a mismatch aborts generation.
"""
import copy
import os
import sys

import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, '_shim'))
sys.path.insert(0, '/root/reference')
sys.path.insert(0, ROOT)

from oracle import fixtures as fx          # noqa: E402
from oracle import genie_oracle as O       # noqa: E402

from genie.module.quantization import LookupFreeQuantization   # noqa: E402  (the reference)
from genie.module.attention import SpaceTimeAttention          # noqa: E402
from genie.module.video import CausalConv3d, VideoResidualBlock, BlurPooling3d  # noqa: E402
from genie.module.video import DepthToSpaceTimeUpsample, SpaceTimeDownsample    # noqa: E402
from genie.module.norm import AdaptiveGroupNorm                 # noqa: E402
from genie.tokenizer import VideoTokenizer                      # noqa: E402
from genie.action import LatentAction                           # noqa: E402
from genie.dynamics import DynamicsModel                        # noqa: E402

OUT = os.path.join(ROOT, 'tests', 'golden')
os.makedirs(OUT, exist_ok=True)
torch.set_num_threads(os.cpu_count())
OUT_SAMPLE = 16384     # values stored per layer output / input gradient: keeps each golden file under 1 MB


class ZeroLoss(nn.Module):
    def forward(self, *a, **k):
        return torch.zeros(())


def load_det(module: nn.Module, gain: float = 1.0):
    """Overwrite every parameter with its closed-form value; keep structural buffers (freq, bit_mask)."""
    shapes = {k: tuple(v.shape) for k, v in module.state_dict().items()}
    sd = O.det_state_dict(shapes, gain)
    missing = module.load_state_dict(sd, strict=False)
    assert all(k.endswith(('freq', 'bit_mask', 'blur')) for k in missing.missing_keys), missing
    return {k: v.detach().clone() for k, v in module.state_dict().items()}


def close(a, b, name, rtol=1e-4, atol=1e-5):
    a, b = torch.as_tensor(a), torch.as_tensor(b)
    if a.dtype.is_floating_point:
        ok = torch.allclose(a.float(), b.float(), rtol=rtol, atol=atol)
        err = (a.float() - b.float()).abs().max().item()
    else:
        ok = torch.equal(a, b)
        err = (a != b).sum().item()
    print(f'  oracle vs reference  {name:34s} {"ok" if ok else "MISMATCH"}  (max err {err:.3e})')
    assert ok, name


def grads_of(module):
    return {k: p.grad.detach().clone() for k, p in module.named_parameters() if p.grad is not None}


def output_entry(key, y, dx, module):
    """Output and input gradient of a layer as OUT_SAMPLE values each (det_sample), its gradients summarized."""
    return {'y': O.det_sample(y, key + '.y', OUT_SAMPLE), 'dx': O.det_sample(dx, key + '.dx', OUT_SAMPLE),
            'grads': summarize_grads(grads_of(module))}


def summarize_grads(g, keep_full=()):
    """Norms for every gradient, full tensors only for the small ones named in keep_full."""
    out = {'norm': {k: v.norm().item() for k, v in g.items()}, 'full': {}}
    for k, v in g.items():
        if k in keep_full or v.numel() <= 4096:
            out['full'][k] = v
    return out


# ------------------------------------------------------------------------------------------------
def gen_kats():
    """Small closed-form facts of the reference (SURVEY.md §8c), re-derived from the reference here."""
    dm = DynamicsModel(desc=fx.bp(fx.MINI_DYN_DESC), **fx.MINI_DYN)
    sched = {w: dm.get_schedule(10, (16, 16), w) for w in ('linear', 'cosine', 'arccos')}
    for w, s in sched.items():
        close(O.maskgit_schedule(10, (16, 16), w), s, f'schedule[{w}]')
    lfq = LookupFreeQuantization(4, input_dim=4).eval()
    x = torch.tensor([[[0.5, -1., 0., 2.], [-.1, -.2, -.3, -.4], [1., 1., 1., 1.]]])
    (q, idx), _ = lfq(x)
    (oq, oidx), _ = O.lfq(x, 4, training=False)
    close(oq, q, 'lfq D=4 quant')
    close(oidx, idx, 'lfq D=4 idxs')
    from genie.module.attention import RotaryEmbedding
    f1 = RotaryEmbedding(8, '1d').freq.detach()
    f2 = RotaryEmbedding(8, '2d').freq.detach()
    close(O.rope_freq(8, '1d'), f1, 'rope freq 1d')
    close(O.rope_freq(8, '2d'), f2, 'rope freq 2d')
    blur = BlurPooling3d(4, 3).blur
    close(O.blur_kernel(3), blur, 'blur kernel')
    xb = O.det_uniform('kat.blur.x', (1, 4, 4, 8, 8))
    close(O.blur_pool3d(xb, 3, 2, 2), BlurPooling3d(4, 3)(xb), 'blur_pool3d')
    torch.save({'schedule': sched, 'lfq4_x': x, 'lfq4_quant': q, 'lfq4_idx': idx, 'bit_mask': lfq.bit_mask,
                'rope_1d_c8': f1, 'rope_2d_c8': f2, 'blur3': blur, 'blur_pool_out': BlurPooling3d(4, 3)(xb)},
               os.path.join(OUT, 'kats.pt'))


def gen_layers():
    """Single-layer vectors: CausalConv3d (stride 1 and strided), residual block, up-sample, AdaGN."""
    out = {}
    x = O.det_uniform('layers.x', (2, 64, 4, 8, 8))
    x.requires_grad_(True)

    m = CausalConv3d(64, 64, 3)
    sd = load_det(m)
    y = m(x); y.square().mean().backward()
    close(O.causal_conv3d(x, sd['conv3d.weight'], sd['conv3d.bias']), y, 'CausalConv3d k3')
    out['causal_conv3d'] = output_entry('layers.causal_conv3d', y, x.grad, m)
    x.grad = None

    m = SpaceTimeDownsample(64, 3, 64, time_factor=2, space_factor=2)
    sd = load_det(m)
    y = m(x); y.square().mean().backward()
    close(O.spacetime_downsample(sd, '', x, 2, 2), y, 'SpaceTimeDownsample')
    out['spacetime_downsample'] = output_entry('layers.spacetime_downsample', y, x.grad, m)
    x.grad = None

    m = VideoResidualBlock(64, 128)
    sd = load_det(m)
    y = m(x); y.square().mean().backward()
    close(O.video_residual_block(sd, '', x), y, 'VideoResidualBlock 64->128')
    out['video_residual'] = output_entry('layers.video_residual', y, x.grad, m)
    x.grad = None

    m = VideoResidualBlock(64, 128, downsample=(2, 2))      # blur-pool variant (README / test blueprints)
    sd = load_det(m)
    y = m(x); y.square().mean().backward()
    close(O.video_residual_block(sd, '', x, downsample=(2, 2)), y, 'VideoResidualBlock downsample')
    out['video_residual_down'] = output_entry('layers.video_residual_down', y, x.grad, m)
    x.grad = None

    m = DepthToSpaceTimeUpsample(64, kernel_size=3, time_factor=2, space_factor=2)
    sd = load_det(m)
    y = m(x); y.square().mean().backward()
    close(O.depth2spacetime_upsample(sd, '', x, 2, 2), y, 'DepthToSpaceTimeUpsample')
    out['depth2spacetime_upsample'] = output_entry('layers.depth2spacetime_upsample', y, x.grad, m)
    x.grad = None

    m = AdaptiveGroupNorm(6, 8, 64)
    sd = load_det(m)
    cond = O.det_uniform('layers.cond', (2, 6, 2, 4, 4)).sign()
    y = m(x, cond); y.square().mean().backward()
    close(O.adaptive_group_norm(sd, '', x, cond, 8), y, 'AdaptiveGroupNorm')
    out['adaptive_group_norm'] = output_entry('layers.adaptive_group_norm', y, x.grad, m)
    x.grad = None
    torch.save(out, os.path.join(OUT, 'layers.pt'))


def gen_lfq():
    out = {}
    for d, n in ((8, 64), (10, 64), (18, 24)):
        m = LookupFreeQuantization(d, input_dim=d)  # input_dim == d  -> no projection (tokenizer, d_codebook=18)
        x = O.det_uniform(f'lfq.x.{d}', (2, n // 2, d), 0.6)
        x.requires_grad_(True)
        m.train()
        (q, idx), loss = m(x)
        (loss + (q * O.det_uniform(f'lfq.gq.{d}', tuple(q.shape))).sum()).backward()
        (oq, oidx), oloss = O.lfq(x, d, training=True)
        close(oq, q, f'lfq D={d} out'); close(oidx, idx, f'lfq D={d} idxs'); close(oloss, loss, f'lfq D={d} loss')
        out[f'd{d}'] = {'n': n, 'out': q.detach(), 'idxs': idx, 'loss': loss.detach(), 'dx': x.grad.clone()}
    torch.save(out, os.path.join(OUT, 'lfq.pt'))


def gen_st_block():
    out = {}
    for transpose, cond_dim, shape in fx.ST_BLOCK_CASES:
        kw = {'time_attn_kw': {'key_dim': cond_dim}} if cond_dim else {}
        m = SpaceTimeAttention(n_head=2, d_head=64, transpose=transpose, **kw)
        sd = load_det(m)
        tag = f't{int(transpose)}_c{cond_dim or 0}'
        x = O.det_uniform(f'st.x.{tag}', shape)
        x.requires_grad_(True)
        t = shape[2] if transpose else shape[1]
        cond = O.det_uniform('st.cond', (2, t, 4)).sign() if cond_dim else None
        y = m(x, cond=(None, cond)) if cond_dim else m(x)
        y.square().mean().backward()
        oy = O.spacetime_attention(sd, '', x, 2, transpose, cond)
        close(oy, y, f'SpaceTimeAttention {tag}', rtol=2e-4, atol=2e-5)
        out[tag] = output_entry(f'st_block.{tag}', y, x.grad, m)
        x.grad = None
    torch.save(out, os.path.join(OUT, 'st_block.pt'))


def gen_tokenizer():
    tok = VideoTokenizer(fx.bp(fx.MINI_ENC), fx.bp(fx.MINI_DEC), d_codebook=fx.MINI_D_CODEBOOK,
                         gan_loss_weight=0, perc_loss_weight=0)
    tok.gan_crit = tok.perc_crit = ZeroLoss()
    sd = load_det(tok)
    video = O.det_uniform('tokenizer.video', fx.MINI_VIDEO_SHAPE)
    quant, idxs = tok.tokenize(video)
    oq, oidx = O.tokenizer_tokenize(sd, fx.MINI_ENC, video, fx.MINI_D_CODEBOOK)
    close(oq, quant, 'tokenize quant'); close(oidx, idxs, 'tokenize idxs')
    dec = tok.decode(quant).detach()
    close(O.tokenizer_decode(sd, fx.MINI_DEC, quant), dec, 'decode', rtol=2e-4, atol=2e-5)
    tok.train()
    loss, (rec_loss, _, _, _, q_loss) = tok(video)
    loss.backward()
    oloss, (orec, oq_loss), orec_v, _ = O.tokenizer_forward(sd, fx.MINI_ENC, fx.MINI_DEC, video, fx.MINI_D_CODEBOOK)
    close(oloss, loss, 'forward loss'); close(orec, rec_loss, 'rec loss'); close(oq_loss, q_loss, 'quant loss')
    enc = tok.encode(video).detach()
    torch.save({'quant': quant, 'idxs': idxs, 'decode': dec, 'enc': enc, 'loss': loss.detach(),
                'rec_loss': rec_loss.detach(), 'quant_loss': q_loss.detach(), 'rec_video': orec_v.detach(),
                'grads': summarize_grads(grads_of(tok)), 'n_params': sum(p.numel() for p in tok.parameters())},
               os.path.join(OUT, 'tokenizer_mini.pt'))


def gen_action_dynamics():
    la = LatentAction(fx.bp(fx.MINI_ACT_ENC), fx.bp(fx.MINI_ACT_DEC), d_codebook=fx.MINI_ACT_D_CODEBOOK,
                      n_embd=fx.MINI_ACT_EMBD, inp_shape=fx.MINI_ACT_VIDEO_SHAPE[-2:])
    la.quant.proj_inp = la.quant.proj_out = nn.Identity()      # constructor omits input_dim (action.py:93-101)
    sd = load_det(la)
    video = O.det_uniform('action.video', fx.MINI_ACT_VIDEO_SHAPE)
    la.train()
    idxs, loss, (rec_loss, q_loss) = la(video)
    loss.backward()
    oidx, oloss, (orec, oq), orecon = O.latent_action_forward(sd, fx.MINI_ACT_ENC, fx.MINI_ACT_DEC, video,
                                                             fx.MINI_ACT_D_CODEBOOK)
    close(oidx, idxs, 'LatentAction idxs'); close(oloss, loss, 'LatentAction loss', rtol=2e-4)
    torch.save({'idxs': idxs, 'loss': loss.detach(), 'rec_loss': rec_loss.detach(), 'q_loss': q_loss.detach(),
                'recon': orecon.detach(), 'grads': summarize_grads(grads_of(la))},
               os.path.join(OUT, 'latent_action_mini.pt'))

    dm = DynamicsModel(desc=fx.bp(fx.MINI_DYN_DESC), **fx.MINI_DYN)
    sd = load_det(dm)
    u = O.det_uniform('dyn.tokens', fx.MINI_DYN_TOKENS_SHAPE) / (3 ** 0.5)          # in (-1, 1)
    tokens = ((u + 1) * 0.5 * fx.MINI_DYN['tok_vocab']).long().clamp(0, fx.MINI_DYN['tok_vocab'] - 1)
    ua = O.det_uniform('dyn.act', fx.MINI_DYN_TOKENS_SHAPE[:2]) / (3 ** 0.5)
    act = ((ua + 1) * 0.5 * fx.MINI_DYN['act_vocab']).long().clamp(0, fx.MINI_DYN['act_vocab'] - 1)
    mask = O.det_uniform('dyn.mask', fx.MINI_DYN_TOKENS_SHAPE) / (3 ** 0.5) < 0.5   # ~75 % masked
    logits, last = dm(tokens, act)
    close(O.dynamics_forward(sd, fx.MINI_DYN_DESC, tokens, act), logits, 'Dynamics logits', rtol=2e-4, atol=2e-5)
    loss = dm.compute_loss(tokens, act, mask=mask)
    loss.backward()
    close(O.dynamics_loss(sd, fx.MINI_DYN_DESC, tokens, act, mask), loss, 'Dynamics loss', rtol=2e-4)
    torch.save({'tokens': tokens, 'act': act, 'mask': mask, 'logits': logits.detach(), 'loss': loss.detach(),
                'grads': summarize_grads(grads_of(dm))}, os.path.join(OUT, 'dynamics_mini.pt'))


def gen_blur2d():
    """BlurPooling2d (genie/module/image.py:43-85, registry name 'blur_pool'): outputs and input gradients."""
    from genie.module.image import BlurPooling2d
    x = O.det_uniform('kat.blur2d.x', (2, 16, 12, 12))
    x.requires_grad_(True)
    out = {}
    for k, s in ((3, 2), (4, 2)):
        m = BlurPooling2d(k, stride=s)
        y = m(x)
        y.backward(O.det_uniform(f'kat.blur2d.g.{k}', tuple(y.shape)))
        out[f'k{k}s{s}'] = {'y': y.detach(), 'dx': x.grad.clone(), 'blur': m.blur.clone()}
        x.grad = None
    torch.save(out, os.path.join(OUT, 'blur2d.pt'))


def gen_gan_perceptual():
    """GAN critic + hinge losses + perceptual loss (genie/module/discriminator.py, loss.py) run by the real reference.
    Test seams: torch.randperm is replaced by fixed permutations (frame picking), VGG16 gets closed-form weights
    (`weights='DEFAULT'` needs a download)."""
    from genie.module.discriminator import FrameDiscriminator
    from genie.module.loss import GANLoss, PerceptualLoss
    out = {}
    disc = FrameDiscriminator(inp_size=32)
    sd = load_det(disc)
    frames = O.det_uniform('gan.frames', (4, 3, 32, 32))
    frames.requires_grad_(True)
    score = disc(frames)
    (-score.mean()).backward()
    out['disc'] = {'score': score.detach(), 'dframes': frames.grad.clone(), 'grads': summarize_grads(grads_of(disc))}
    # hinge losses through GANLoss with fixed frame picks
    b, t, k = 2, 8, 2
    perms = [torch.tensor([3, 0, 5, 1, 7, 2, 6, 4]), torch.tensor([6, 2, 1, 7, 0, 4, 3, 5])]
    idxs = torch.cat([p[:k] for p in perms])
    real_randperm = torch.randperm

    def fixed_perms():
        it = iter(perms * 8)
        return lambda n, **kw: next(it)

    gan = GANLoss(discriminate='frames', num_frames=k, inp_size=32)
    gan.disc.load_state_dict(sd)
    rec = O.det_uniform('gan.rec', (b, 3, t, 32, 32))
    rec.requires_grad_(True)
    inp = O.det_uniform('gan.inp', (b, 3, t, 32, 32))
    torch.randperm = fixed_perms()
    try:
        gen_loss = gan(rec, inp, train_gen=True)
        torch.randperm = fixed_perms()
        dis_loss = gan(rec, inp, train_gen=False)
    finally:
        torch.randperm = real_randperm
    (gen_loss + dis_loss).backward()
    out['gan'] = {'frames_idxs': idxs, 'gen_loss': gen_loss.detach(), 'dis_loss': dis_loss.detach(),
                  'drec': rec.grad.clone(), 'grads': summarize_grads(grads_of(gan))}
    # the 3-D critic (gan_discriminate='video')
    from genie.module.discriminator import VideoDiscriminator
    vd = VideoDiscriminator(inp_size=(8, 32, 32))
    load_det(vd)
    clip = O.det_uniform('gan.clip', (2, 3, 8, 32, 32))
    clip.requires_grad_(True)
    vs = vd(clip)
    (-vs.mean()).backward()
    out['video_disc'] = {'score': vs.detach(), 'dclip': clip.grad.clone(), 'grads': summarize_grads(grads_of(vd))}
    # perceptual loss, closed-form VGG16 feature weights
    perc = PerceptualLoss(model_weights=None, num_frames=k)
    vsd = O.det_state_dict({k_: tuple(v.shape) for k_, v in perc.percept_model.state_dict().items()
                            if k_.startswith('features')}, gain=1.4)
    perc.percept_model.load_state_dict(vsd, strict=False)
    torch.randperm = fixed_perms()
    try:
        with torch.no_grad():
            pl = perc(rec.detach(), inp)
    finally:
        torch.randperm = real_randperm
    assert not pl.requires_grad
    out['perc'] = {'frames_idxs': idxs, 'loss': pl.detach()}
    print(f'  gan: gen {gen_loss.item():.5f} dis {dis_loss.item():.5f}; perceptual {pl.item():.6f}')
    torch.save(out, os.path.join(OUT, 'gan_perceptual.pt'))


def gen_generate():
    """DynamicsModel.generate run by the REAL reference with two test seams: torch.multinomial is replaced by the
    inverse-CDF draw on injected uniforms (O.inverse_cdf_draw) and, for the big case, forward() returns given logits."""
    out = {}
    real_multinomial = torch.multinomial

    def run(dm, tokens, act, steps, uniforms):
        it = iter(uniforms)
        torch.multinomial = lambda prob, num_samples=1, **kw: O.inverse_cdf_draw(prob, next(it))
        try:
            return dm.generate(tokens, act, steps=steps)
        finally:
            torch.multinomial = real_multinomial

    # (1) the mini model end to end (P = 64 positions, V = 64)
    dm = DynamicsModel(desc=fx.bp(fx.MINI_DYN_DESC), **fx.MINI_DYN)
    load_det(dm)
    b, t, h, w = 2, 3, 8, 8
    u = O.det_uniform('gen.tokens', (b, t, h, w)) / (3 ** 0.5)
    tokens = ((u + 1) * 0.5 * fx.MINI_DYN['tok_vocab']).long().clamp(0, fx.MINI_DYN['tok_vocab'] - 1)
    ua = O.det_uniform('gen.act', (b, t)) / (3 ** 0.5)
    act = ((ua + 1) * 0.5 * fx.MINI_DYN['act_vocab']).long().clamp(0, fx.MINI_DYN['act_vocab'] - 1)
    steps = 5
    uni = (O.det_uniform('gen.uniforms', (steps, b * h * w)) / (3 ** 0.5) + 1) * 0.5
    with torch.no_grad():
        tok_id = torch.cat([tokens, torch.zeros(b, 1, h, w, dtype=tokens.dtype)], 1)
        act_id = torch.cat([act, torch.zeros(b, 1, dtype=act.dtype)], 1)
        _, logits_last = dm(tok_id, act_id)
    pred = run(dm, tokens, act, steps, uni)
    sched = dm.get_schedule(steps, (h, w))
    close(O.maskgit_generate(logits_last, tokens, uni, sched), pred, 'generate (mini model)')
    out['mini'] = {'tokens': tokens, 'act': act, 'steps': steps, 'uniforms': uni, 'logits_last': logits_last,
                   'pred_tok': pred}
    # (2) configs[3] sizes: P = 256 positions, V = 1024, 25 steps (Genie.forward's steps_per_frame) on given logits
    b, t, h, w, V, steps = 2, 2, 16, 16, 1024, 25
    logits = O.det_uniform('gen.big.logits', (b, h, w, V), 2.0)
    tokens = ((O.det_uniform('gen.big.tokens', (b, t, h, w)) / (3 ** 0.5) + 1) * 0.5 * V).long().clamp(0, V - 1)
    act = torch.zeros(b, t, dtype=torch.long)
    uni = (O.det_uniform('gen.big.uniforms', (steps, b * h * w)) / (3 ** 0.5) + 1) * 0.5
    dm.forward = lambda tok_id, act_id: (None, logits)
    for which in ('linear', 'cosine'):
        it = iter(uni)
        torch.multinomial = lambda prob, num_samples=1, **kw: O.inverse_cdf_draw(prob, next(it))
        try:
            pred = dm.generate(tokens, act, steps=steps, which=which)
        finally:
            torch.multinomial = real_multinomial
        sched = dm.get_schedule(steps, (h, w), which)
        close(O.maskgit_generate(logits, tokens, uni, sched), pred, f'generate (given logits, {which})')
        out[f'big_{which}'] = {'tokens': tokens, 'steps': steps, 'pred_tok': pred}
    torch.save(out, os.path.join(OUT, 'generate.pt'))


PLATFORMER_SAMPLE = 8192


def gen_platformer():
    """The reference's Platformer2D on the clips of fixtures.write_platformer_clips: for every output format and padding,
    each clip's shape and a det_sample of its values, stored x 255 as uint8 (the frames are uint8 / 255, so exactly)."""
    import shutil
    import tempfile
    from genie.module.data import Platformer2D
    root = tempfile.mkdtemp(prefix='platformer_')
    try:
        fx.write_platformer_clips(root)
        out = {}
        for fmt in ('t c h w', 'c t h w'):
            for padding in ('none', 'repeat', 'zero'):
                ds = Platformer2D(root, split='train', padding=padding, num_frames=16, output_format=fmt)
                for i, f in enumerate(ds.file_names):
                    name = os.path.basename(f)
                    v = O.det_sample(ds[i], f'platformer.{fmt}.{padding}.{name}', PLATFORMER_SAMPLE)
                    u8 = (v * 255.).round().to(torch.uint8)
                    assert torch.equal(u8.float() / 255., v)
                    out[(fmt, padding, name)] = {'shape': tuple(ds[i].shape), 'x255': u8}
    finally:
        shutil.rmtree(root)
    torch.save(out, os.path.join(OUT, 'platformer.pt'))


if __name__ == '__main__':
    if sys.argv[1:] == ['generate']:
        with torch.no_grad():
            gen_generate()
        sys.exit(0)
    if sys.argv[1:] == ['platformer']:
        gen_platformer()
        sys.exit(0)
    if sys.argv[1:] == ['gan']:
        gen_gan_perceptual()
        sys.exit(0)
    with torch.no_grad():
        gen_kats()
        gen_generate()
    gen_blur2d()
    gen_gan_perceptual()
    gen_layers()
    gen_lfq()
    gen_st_block()
    gen_tokenizer()
    gen_action_dynamics()
    gen_platformer()
    sizes = {f: os.path.getsize(os.path.join(OUT, f)) for f in sorted(os.listdir(OUT))}
    print('golden files:', sizes, 'total', sum(sizes.values()))
