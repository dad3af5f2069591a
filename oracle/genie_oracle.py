"""oracle/genie_oracle.py — CPU restatement of open-genie's hot path.   *** TEST INFRASTRUCTURE ***

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may import this.
The product (open_genie_b200) never does: it fails loudly when its CUDA library is missing.

What this is
    A functional, fp32, torch-CPU restatement of the reference modules on the path named by
    BASELINE.json (VideoTokenizer encode -> LFQ -> decode, space-time attention blocks, LatentAction,
    DynamicsModel).  The reference's arithmetic lives in third-party PyTorch ATen calls
    (requirements.txt pins torch==2.3.0; 2.11.0 is what this image has), so the restatement calls the
    same ATen primitives (conv3d, group_norm, layer_norm, scaled_dot_product_attention, softmax ...)
    directly on a reference-format ``state_dict`` instead of going through the reference's nn.Modules.
    Every function cites the reference file:line it follows (paths relative to the reference repo).

Pinning
    The reference's own tests hold no value-level vectors (SURVEY.md §4), so this oracle is pinned
    against outputs of the reference itself, imported from /root/reference in the build container by
    oracle/make_golden.py; the resulting vectors are committed under tests/golden/ and checked by
    tests/test_oracle_golden.py (CPU).  Parity status: PINNED against reference outputs.
"""
from __future__ import annotations

import math
from typing import Dict, List, Sequence, Tuple

import torch
import torch.nn.functional as F
from torch import Tensor

StateDict = Dict[str, Tensor]


# ------------------------------------------------------------------------------------------------
# deterministic, RNG-free tensors (shared by make_golden.py, the tests, smoke() and bench.py)
# ------------------------------------------------------------------------------------------------
def _key_seed(key: str) -> int:
    h = 1469598103934665603  # FNV-1a
    for ch in key.encode():
        h = ((h ^ ch) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def det_uniform(key: str, shape: Sequence[int], scale: float = 1.0) -> Tensor:
    """Closed-form pseudo-random tensor in (-scale*sqrt(3), scale*sqrt(3)) (std == scale).

    Pure integer arithmetic (splitmix64 over the flat index), so every machine and every torch version
    produces the same bits — unlike torch.manual_seed streams."""
    import numpy as np

    n = int(math.prod(shape)) if len(shape) else 1
    with np.errstate(over='ignore'):
        z = np.arange(n, dtype=np.uint64) + np.uint64(_key_seed(key))
        z = (z + np.uint64(0x9E3779B97F4A7C15))
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    u = (z >> np.uint64(11)).astype(np.float64) / float(1 << 53)
    v = (u * 2.0 - 1.0) * (scale * math.sqrt(3.0))
    return torch.from_numpy(v.astype(np.float32)).reshape(tuple(shape))


def det_indices(key: str, numel: int, n: int = 1024) -> Tensor:
    """n deterministic flat indices into a tensor of `numel` elements (all of them when numel <= n): the sample
    on which the full-size goldens store / compare big gradients."""
    if numel <= n:
        return torch.arange(numel)
    u = det_uniform('idx.' + key, (n,)) / math.sqrt(3.0)           # (-1, 1)
    return ((u.double() + 1.0) * 0.5 * numel).long().clamp_(0, numel - 1)


def det_sample(t: Tensor, key: str, n: int = 1024) -> Tensor:
    """The flattened values of `t` at det_indices(key, t.numel(), n): how the goldens store big tensors. A stored
    sample of m values is matched by det_sample(got, key, m), whether or not it holds the whole tensor."""
    flat = t.detach().flatten()
    return flat[det_indices(key, flat.numel(), n).to(flat.device)]


def det_state_dict(shapes: Dict[str, Sequence[int]], gain: float = 1.0) -> StateDict:
    """Deterministic weights for a reference-format state_dict (shapes from the reference module).

    conv / linear weights ~ U with std gain/sqrt(fan_in); biases small; norm weights near 1;
    RoPE ``freq`` and LFQ ``bit_mask`` are structural and must be supplied by the caller instead."""
    sd: StateDict = {}
    for k, shp in shapes.items():
        shp = tuple(shp)
        if k.endswith('freq') or k.endswith('bit_mask') or k.endswith('blur'):
            continue
        if k.endswith('weight') and len(shp) >= 2:
            fan_in = int(math.prod(shp[1:]))
            sd[k] = det_uniform(k, shp, gain / math.sqrt(fan_in))
        elif k.endswith('weight'):  # norm gains
            sd[k] = 1.0 + det_uniform(k, shp, 0.1)
        else:  # biases
            sd[k] = det_uniform(k, shp, 0.05)
    return sd


# ------------------------------------------------------------------------------------------------
# genie/module/video.py
# ------------------------------------------------------------------------------------------------
def causal_conv3d(x: Tensor, weight: Tensor, bias: Tensor | None, stride=(1, 1, 1), dilation=(1, 1, 1)) -> Tensor:
    """CausalConv3d.forward — video.py:154-164 (padding) and 178-192 (pad + conv3d).

    time pad (front only) = (kt-1)*dil_t + (1 - stride_t); space pad = (k-1)//2 on both sides."""
    kt, kh, kw = weight.shape[2:]
    pt = (kt - 1) * dilation[0] + (1 - stride[0])
    ph, pw = (kh - 1) // 2, (kw - 1) // 2
    x = F.pad(x, (pw, pw, ph, ph, pt, 0), mode='constant')
    return F.conv3d(x, weight, bias, stride=stride, dilation=dilation)


def blur_kernel(k: int = 3) -> Tensor:
    """get_blur_kernel — video.py:22-56: outer product of Pascal rows, normalised to sum 1."""
    row = torch.tensor([math.comb(k - 1, i) for i in range(k)], dtype=torch.float32)
    ker = row[:, None, None] * row[None, :, None] * row[None, None, :]
    return ker / ker.sum()


def blur_pool3d(x: Tensor, k: int, time_factor: int, space_factor: int, num_groups: int = 1,
                out_channels: int | None = None) -> Tensor:
    """BlurPooling3d.forward — video.py:514-534. With num_groups == 1 the repeated kernel makes this a
    dense conv whose every tap is the same blur, i.e. out[:, o] = blur(sum_c x[:, c]) for every o."""
    c = x.shape[1]
    o = out_channels if out_channels is not None else c
    ker = blur_kernel(k).to(x)[None, None].expand(o, c // num_groups, k, k, k)
    pad = (k - 1) // 2
    return F.conv3d(x, ker, stride=(time_factor, space_factor, space_factor), padding=pad, groups=num_groups)


def video_residual_block(sd: StateDict, pre: str, x: Tensor, num_groups: int = 1, downsample=None) -> Tensor:
    """VideoResidualBlock.forward as built by the MAGVIT2 blueprints (use_causal=False) — video.py:597-631
    (layers) and 648 (main(x) + res(x)); `downsample=(tf, sf)` adds the BlurPooling3d of both branches (589-621).

    main = GN(num_groups) -> SiLU -> Conv3d(k3,p1) -> [blur] -> GN -> SiLU -> Conv3d(k3,p1); res = [blur] -> Conv3d(k1)."""
    h = F.group_norm(x, num_groups, sd[pre + 'main.0.weight'], sd[pre + 'main.0.bias'], 1e-5)
    h = F.silu(h)
    w = sd[pre + 'main.2.weight']
    h = F.conv3d(h, w, sd[pre + 'main.2.bias'], padding=tuple((k - 1) // 2 for k in w.shape[2:]))
    if downsample is not None:
        h = blur_pool3d(h, w.shape[2], downsample[0], downsample[1], num_groups)
        x = blur_pool3d(x, w.shape[2], downsample[0], downsample[1], num_groups)
    h = F.group_norm(h, num_groups, sd[pre + 'main.4.weight'], sd[pre + 'main.4.bias'], 1e-5)
    h = F.silu(h)
    w = sd[pre + 'main.6.weight']
    h = F.conv3d(h, w, sd[pre + 'main.6.bias'], padding=tuple((k - 1) // 2 for k in w.shape[2:]))
    r = F.conv3d(x, sd[pre + 'res.1.weight'], sd[pre + 'res.1.bias'])
    return h + r


def spacetime_downsample(sd: StateDict, pre: str, x: Tensor, time_factor: int, space_factor: int) -> Tensor:
    """SpaceTimeDownsample — video.py:457-483: a strided CausalConv3d."""
    return causal_conv3d(x, sd[pre + 'go_down.conv3d.weight'], sd.get(pre + 'go_down.conv3d.bias'),
                         stride=(time_factor, space_factor, space_factor))


def depth2spacetime_upsample(sd: StateDict, pre: str, x: Tensor, time_factor: int, space_factor: int) -> Tensor:
    """DepthToSpaceTimeUpsample — video.py:397-409: CausalConv3d to C*tf*sf^2 channels, then
    'b (c p q r) t h w -> b c (t p) (h q) (w r)'."""
    y = causal_conv3d(x, sd[pre + 'go_up.0.conv3d.weight'], sd.get(pre + 'go_up.0.conv3d.bias'))
    b, cc, t, h, w = y.shape
    p, q, r = time_factor, space_factor, space_factor
    c = cc // (p * q * r)
    y = y.reshape(b, c, p, q, r, t, h, w).permute(0, 1, 5, 2, 6, 3, 7, 4)
    return y.reshape(b, c, t * p, h * q, w * r)


# ------------------------------------------------------------------------------------------------
# genie/module/norm.py
# ------------------------------------------------------------------------------------------------
def adaptive_group_norm(sd: StateDict, pre: str, x: Tensor, cond: Tensor, num_groups: int, eps: float = 1e-5) -> Tensor:
    """AdaptiveGroupNorm.forward — norm.py:55-69: GN(x) * Linear_std(mean(cond)) + Linear_avg(mean(cond))."""
    y = F.group_norm(x, num_groups, sd[pre + 'weight'], sd[pre + 'bias'], eps)
    c = cond.flatten(2).mean(-1)
    std = F.linear(c, sd[pre + 'std.weight'], sd[pre + 'std.bias'])
    avg = F.linear(c, sd[pre + 'avg.weight'], sd[pre + 'avg.bias'])
    view = (x.shape[0], x.shape[1]) + (1,) * (x.dim() - 2)
    return y * std.view(view) + avg.view(view)


# ------------------------------------------------------------------------------------------------
# genie/module/quantization.py
# ------------------------------------------------------------------------------------------------
def lfq_bit_mask(d: int) -> Tensor:
    """quantization.py:72 — MSB-first powers of two."""
    return 2 ** torch.arange(d - 1, -1, -1)


def lfq_codebook(d: int) -> Tensor:
    """quantization.py:74-75 — all 2^d sign codes, row j = bits of j (MSB first) mapped to {-1,+1}."""
    codes = torch.arange(2 ** d)[:, None] & lfq_bit_mask(d)
    return 2 * (codes != 0).float() - 1


def lfq_entropy(p: Tensor, eps: float = 1e-6) -> Tensor:
    """entropy — quantization.py:17-28."""
    return -(p * torch.log(p.clamp(min=eps))).sum(dim=-1)


def lfq(x: Tensor, d: int, training: bool, beta: float = 100., transpose: bool = False,
        commit_weight: float = .25, entropy_weight: float = .1, diversity_weight: float = 1.,
        proj_inp: Tuple[Tensor, Tensor | None] | None = None,
        proj_out: Tuple[Tensor, Tensor | None] | None = None):
    """LookupFreeQuantization.forward (num_codebook == 1) — quantization.py:77-133.

    Returns ((out, idxs), loss-or-None). ``idxs`` keeps the reference's ``.squeeze()`` (line 110)."""
    inp = x.movedim(1, -1) if transpose else x                     # 'b d ... -> b ... d'      (84)
    lead = inp.shape[1:-1]
    inp = inp.reshape(inp.shape[0], -1, inp.shape[-1])             # pack 'b * d'              (85)
    if proj_inp is not None:
        inp = F.linear(inp, proj_inp[0], proj_inp[1])              #                           (87)
    inp = inp.unsqueeze(2)                                         # 'b n (c d) -> b n c d'    (90)
    quant = inp.sign()                                             #                           (97)
    idxs = ((inp > 0).int() * lfq_bit_mask(d).int()).sum(-1)       #                           (98)
    code = (inp + (quant - inp).detach()) if training else quant   # STE                       (101)
    code = code.flatten(2)
    out = code if proj_out is None else F.linear(code, proj_out[0], proj_out[1])   #           (105)
    out = out.reshape(out.shape[0], *lead, out.shape[-1])
    out = out.movedim(-1, 1) if transpose else out
    idxs = idxs.reshape(idxs.shape[0], *lead, 1).squeeze()         #                           (110)
    if not training:
        return (out, idxs), None
    logits = 2 * torch.einsum('bncd,jd->bncj', inp, lfq_codebook(d).to(inp))       #           (116)
    prob = (logits * beta).softmax(dim=-1)                         #                           (117)
    prob = prob.flatten(0, 1)                                      #                           (118)
    avg_prob = prob.mean(dim=0)                                    #                           (120)
    inp_ent = lfq_entropy(prob).mean()
    avg_ent = lfq_entropy(avg_prob).mean()
    entropy_loss = inp_ent + diversity_weight * avg_ent            # NB: '+' as in the reference (125)
    commit = F.mse_loss(inp, quant.detach())                       #                           (128)
    return (out, idxs), entropy_loss * entropy_weight + commit * commit_weight     #           (131)


# ------------------------------------------------------------------------------------------------
# genie/module/attention.py
# ------------------------------------------------------------------------------------------------
def rope_freq(dim: int, kind: str) -> Tensor:
    """RotaryEmbedding.__init__ — attention.py:31-39."""
    if kind == '1d':
        return 1. / (10000 ** (torch.arange(0, dim, 2)[:dim // 2].float() / dim))
    if kind == '2d':
        return torch.linspace(1., 10 / 2, dim // 2) * math.pi
    raise ValueError(kind)


def rope(x: Tensor, freq: Tensor) -> Tensor:
    """RotaryEmbedding.forward/apply — attention.py:48-94, for (B, n, C) input: interleaved-pair rotation
    over the FULL channel dim, angle[n, 2i] = angle[n, 2i+1] = n * freq[i]."""
    n = x.shape[-2]
    ang = torch.arange(n, dtype=freq.dtype)[:, None] * freq[None, :]
    ang = ang.repeat_interleave(2, dim=-1)
    x1, x2 = x[..., 0::2], x[..., 1::2]
    rot = torch.stack((-x2, x1), dim=-1).flatten(-2)
    return (x * ang.cos() + rot * ang.sin()).type(x.dtype)


def attention_core(sd: StateDict, pre: str, x: Tensor, n_head: int, causal: bool, kind: str,
                   cond: Tensor | None = None) -> Tensor:
    """Attention.forward — attention.py:199-239, in the HEAD-valid configuration where
    d_inp == n_head*d_head, so to_q (and to_k/to_v without cond) are Identity:
    q = k = v = LayerNorm(RoPE(x)); scale = n_head * d_head**-0.5 (line 195's precedence)."""
    c = x.shape[-1]
    d_head = c // n_head
    q = rope(x, sd[pre + 'embed.freq'])
    q = F.layer_norm(q, (c,), sd[pre + 'norm.weight'], sd[pre + 'norm.bias'], 1e-5)
    if cond is None:
        k = v = q
    else:  # key = cond; val = key (line 224-225); Linear(key_dim -> C, bias=False) each (127-129)
        k = F.linear(cond, sd[pre + 'to_qkv.to_k.weight'])
        v = F.linear(cond, sd[pre + 'to_qkv.to_v.weight'])

    def split(t):  # 'n (h d) -> h n d'
        return t.reshape(t.shape[0], t.shape[1], n_head, d_head).transpose(1, 2)

    o = F.scaled_dot_product_attention(split(q), split(k), split(v), is_causal=causal,
                                       scale=n_head * d_head ** -0.5)
    return o.transpose(1, 2).reshape(x.shape[0], x.shape[1], c)     # 'b h n d -> b n (h d)'


def spatial_attention(sd: StateDict, pre: str, video: Tensor, n_head: int, transpose: bool) -> Tensor:
    """SpatialAttention.forward — attention.py:279-307 (cond path is dead code at HEAD)."""
    x = video.movedim(1, -1) if transpose else video               # -> b t h w c
    b, t, h, w, c = x.shape
    o = attention_core(sd, pre, x.reshape(b * t, h * w, c), n_head, False, '2d')
    o = o.reshape(b, t, h, w, c)
    return o.movedim(-1, 1) if transpose else o


def temporal_attention(sd: StateDict, pre: str, video: Tensor, n_head: int, transpose: bool,
                       cond: Tensor | None = None) -> Tensor:
    """TemporalAttention.forward — attention.py:347-371; causal; cond (b,t,k) repeated over (h,w)."""
    x = video.movedim(1, -1) if transpose else video               # b t h w c
    b, t, h, w, c = x.shape
    x = x.permute(0, 2, 3, 1, 4).reshape(b * h * w, t, c)
    if cond is not None:
        cond = cond[:, None, None].expand(b, h, w, *cond.shape[1:]).reshape(b * h * w, *cond.shape[1:])
    o = attention_core(sd, pre, x, n_head, True, '1d', cond)
    o = o.reshape(b, h, w, t, c).permute(0, 3, 1, 2, 4)
    return o.movedim(-1, 1) if transpose else o


def spacetime_attention(sd: StateDict, pre: str, video: Tensor, n_head: int, transpose: bool,
                        time_cond: Tensor | None = None) -> Tensor:
    """SpaceTimeAttention.forward — attention.py:456-474, skips all Identity (d_inp/d_out unset):
    x = space(x)+x ; x = time(x,cond)+x ; x = ffn(x)+x with
    ffn = GN(n_head, C) -> Conv3d(C, C, 3, padding=1, bias=False) (attention.py:429-444, misc.py:92-98)."""
    x = spatial_attention(sd, pre + 'space_attn.', video, n_head, transpose) + video
    x = temporal_attention(sd, pre + 'temp_attn.', x, n_head, transpose, time_cond) + x
    y = x if transpose else x.movedim(-1, 1)                       # Rearrange -> b c t h w
    y = F.group_norm(y, n_head, sd[pre + 'ffn.1.net.0.weight'], sd[pre + 'ffn.1.net.0.bias'], 1e-5)
    y = F.conv3d(y, sd[pre + 'ffn.1.net.1.0.weight'], None, padding=1)
    y = y if transpose else y.movedim(1, -1)
    return y + x


# ------------------------------------------------------------------------------------------------
# blueprint interpreter (genie/module/__init__.py:71-93) + VideoTokenizer (genie/tokenizer.py)
# ------------------------------------------------------------------------------------------------
def expand_blueprint(bp) -> List[Tuple[str, dict]]:
    """parse_blueprint's expansion of n_rep / has_ext — module/__init__.py:77-91 — without mutating bp."""
    out = []
    for desc in bp:
        if isinstance(desc, str):
            desc = (desc, {})
        name, kw = desc
        kw = dict(kw)
        rep = kw.pop('n_rep', 1)
        out.extend([(name, dict(kw))] * rep)
    return out


def run_layers(sd: StateDict, prefix: str, bp, x: Tensor, cond: Tensor | None = None) -> Tensor:
    """The layer loop of VideoTokenizer.encode / decode — tokenizer.py:313-317, 326-330."""
    for i, (name, kw) in enumerate(expand_blueprint(bp)):
        pre = f'{prefix}.{i}.'
        if name == 'causal-conv3d':
            x = causal_conv3d(x, sd[pre + 'conv3d.weight'], sd.get(pre + 'conv3d.bias'))
        elif name == 'video-residual':
            x = video_residual_block(sd, pre, x, kw.get('num_groups', 1))
        elif name == 'spacetime_downsample':
            x = spacetime_downsample(sd, pre, x, kw.get('time_factor', 2), kw.get('space_factor', 2))
        elif name == 'depth2spacetime_upsample':
            x = depth2spacetime_upsample(sd, pre, x, kw.get('time_factor', 2), kw.get('space_factor', 2))
        elif name == 'group_norm':
            x = F.group_norm(x, kw['num_groups'], sd[pre + 'weight'], sd[pre + 'bias'], 1e-5)
        elif name == 'adaptive_group_norm':
            x = adaptive_group_norm(sd, pre, x, cond, kw['num_groups'])
        elif name == 'silu':
            x = F.silu(x)
        elif name == 'space-time_attn':
            tc = cond if kw.get('has_ext', False) else None
            x = spacetime_attention(sd, pre, x, kw['n_head'], kw.get('transpose', False), tc)
        else:
            raise ValueError(f'oracle: module {name!r} is outside the hot-path scope')
    return x


def _lfq_proj(sd: StateDict, which: str):
    k = f'quant.{which}.weight'
    return (sd[k], sd.get(f'quant.{which}.bias')) if k in sd else None


def tokenizer_encode(sd: StateDict, enc_bp, video: Tensor) -> Tensor:
    """VideoTokenizer.encode — tokenizer.py:307-317."""
    return run_layers(sd, 'enc_layers', enc_bp, video)


def tokenizer_decode(sd: StateDict, dec_bp, quant: Tensor, cond: Tensor | None = None) -> Tensor:
    """VideoTokenizer.decode — tokenizer.py:319-330 (cond defaults to the quantised latent)."""
    return run_layers(sd, 'dec_layers', dec_bp, quant, quant if cond is None else cond)


def tokenizer_tokenize(sd: StateDict, enc_bp, video: Tensor, d_codebook: int, beta: float = 100.):
    """VideoTokenizer.tokenize — tokenizer.py:332-350 (eval-mode LFQ: code = sign(x), no loss)."""
    enc = tokenizer_encode(sd, enc_bp, video)
    (q, idxs), _ = lfq(enc, d_codebook, training=False, beta=beta, transpose=True,
                       proj_inp=_lfq_proj(sd, 'proj_inp'), proj_out=_lfq_proj(sd, 'proj_out'))
    return q, idxs


def tokenizer_forward(sd: StateDict, enc_bp, dec_bp, video: Tensor, d_codebook: int, beta: float = 100.,
                      quant_loss_weight: float = 1., **lfq_kw):
    """VideoTokenizer.forward in training mode with the GAN / perceptual terms at zero weight
    (the HEAD-valid configuration of SURVEY.md §8) — tokenizer.py:352-387.
    Returns (loss, (rec_loss, quant_loss), rec_video, idxs)."""
    enc = tokenizer_encode(sd, enc_bp, video)
    (q, idxs), q_loss = lfq(enc, d_codebook, training=True, beta=beta, transpose=True,
                            proj_inp=_lfq_proj(sd, 'proj_inp'), proj_out=_lfq_proj(sd, 'proj_out'), **lfq_kw)
    rec = tokenizer_decode(sd, dec_bp, q)
    rec_loss = F.mse_loss(rec, video)
    loss = rec_loss + q_loss * quant_loss_weight                   # gen/dis/perc terms are 0 (375-379)
    return loss, (rec_loss, q_loss), rec, idxs


# ------------------------------------------------------------------------------------------------
# genie/action.py, genie/dynamics.py
# ------------------------------------------------------------------------------------------------
def latent_action_forward(sd: StateDict, enc_bp, dec_bp, video: Tensor, d_codebook: int,
                          quant_loss_weight: float = 1.):
    """LatentAction.forward — action.py:111-176 with the pinned fix of SURVEY.md §8 (quant.proj_* are
    Identity). Returns (idxs, loss, (rec_loss, q_loss), recon)."""
    x = causal_conv3d(video, sd['proj_in.conv3d.weight'], sd['proj_in.conv3d.bias'])        # 118
    x = run_layers(sd, 'enc_layers', enc_bp, x)                                               # 120-121
    b, c, t = x.shape[:3]
    act = x.movedim(1, 2).reshape(b, t, -1)                        # 'b c t ... -> b t (c ...)'  (84)
    act = F.linear(act, sd['to_act.1.weight'])                     #                             (85-89)
    (q_act, idxs), q_loss = lfq(act, d_codebook, training=True, transpose=False)             # 127
    y = run_layers(sd, 'dec_layers', dec_bp, x, q_act)             # cond = (None, q_act)         (138-145)
    recon = causal_conv3d(y, sd['proj_out.conv3d.weight'], sd['proj_out.conv3d.bias'])       # 147
    rec_loss = F.mse_loss(recon, video)                            #                             (166)
    loss = rec_loss + q_loss * quant_loss_weight                   #                             (170-171)
    return idxs, loss, (rec_loss, q_loss), recon


def dynamics_forward(sd: StateDict, bp, tokens: Tensor, act_id: Tensor) -> Tensor:
    """DynamicsModel.forward — dynamics.py:44-64: tok_emb + act_emb -> ST blocks -> head."""
    x = F.embedding(tokens, sd['tok_emb.weight']) + F.embedding(act_id, sd['act_emb.0.weight'])[:, :, None, None]
    x = run_layers(sd, 'dec_layers', bp, x)
    return F.linear(x, sd['head.weight'], sd['head.bias'])


def dynamics_loss(sd: StateDict, bp, tokens: Tensor, act_id: Tensor, mask: Tensor, fill: int = 0) -> Tensor:
    """DynamicsModel.compute_loss — dynamics.py:66-99 with an explicit mask. NB the target is taken from
    the ALREADY-masked tokens (lines 83, 90), i.e. it is the constant ``fill``."""
    toks = tokens.masked_fill(mask, fill)
    logits = dynamics_forward(sd, bp, toks, act_id)
    m = mask.squeeze()
    return F.cross_entropy(logits[m].reshape(-1, logits.shape[-1]), toks[m].reshape(-1))


def maskgit_schedule(steps: int, shape: Tuple[int, int], which: str = 'linear') -> Tensor:
    """DynamicsModel.get_schedule — dynamics.py:167-194."""
    n = math.prod(shape)
    t = torch.linspace(1, 0, steps)
    if which == 'linear':
        s = 1 - t
    elif which == 'cosine':
        s = torch.cos(t * math.pi * .5)
    elif which == 'arccos':
        s = torch.acos(t) / (math.pi * .5)
    else:
        raise ValueError(f'Unknown schedule type: {which}')
    sch = ((s / s.sum()) * n).round().int().clamp(min=1)
    sch[-1] += n - sch.sum()
    return sch


def inverse_cdf_draw(prob: Tensor, u: Tensor) -> Tensor:
    """Stand-in for torch.multinomial(prob, 1) with INJECTED uniforms (the parity tests patch it into the reference's
    loop too): index of the first element whose running sum exceeds u * total. prob (rows, V), u (rows,) -> (rows, 1)."""
    cdf = prob.float().cumsum(-1)
    tgt = (u.float() * cdf[:, -1])[:, None]
    return (cdf <= tgt).sum(-1, keepdim=True).clamp_(max=prob.shape[-1] - 1)


def maskgit_generate(logits_last: Tensor, tokens: Tensor, uniforms: Tensor, schedule: Tensor, temp: float = 1.,
                     masked_tok: int = 0) -> Tensor:
    """DynamicsModel.generate — dynamics.py:101-165, with the model evaluation factored out: the reference packs
    tok_id = [tokens, code] ONCE before the loop (128) and never refreshes it (pred_tok on line 163 is only the return
    value), so `self(tok_id, act_id)` (140) yields the same last-frame logits `logits_last` (b,h,w,V) every iteration.
    uniforms (steps, b*h*w) replace torch.multinomial's internal randomness (145)."""
    b, t, h, w = tokens.shape
    mask = torch.ones(b, h, w, dtype=torch.bool)                        # 122
    code = torch.full((b, h, w), masked_tok, dtype=tokens.dtype)        # 123
    pred_tok = torch.cat([tokens, code[:, None]], dim=1)
    for s, num_tokens in enumerate(schedule.tolist()):
        if mask.sum() == 0:                                             # 137
            break
        prob = torch.softmax(logits_last / temp, dim=-1).reshape(-1, logits_last.shape[-1])     # 143-144
        pred = inverse_cdf_draw(prob, uniforms[s])                      # 145
        conf = torch.gather(prob, -1, pred).reshape(b, h, w)            # 146-147
        conf[~mask] = -math.inf                                         # 151
        idxs = torch.topk(conf.view(b, -1), k=num_tokens, dim=-1).indices   # 152
        pred = pred.view(b, -1)
        code = code.view(b, -1).scatter(1, idxs, torch.gather(pred, -1, idxs).to(code.dtype)).view(b, h, w)   # 158-159
        mask = mask.view(b, -1).scatter(1, idxs, False).view(b, h, w)   # 160
        pred_tok = torch.cat([tokens, code[:, None]], dim=1)            # 163
    assert mask.sum() == 0
    return pred_tok
