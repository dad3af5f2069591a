#!/usr/bin/env python
"""bench.py — VideoTokenizer train-step frames/sec @ 16x64x64 (BASELINE.json's metric, configs[1]).

    python bench.py --gpus N --steps K --warmup W                 # our arm (one process per GPU via torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K --warmup W  # the reference itself on the host CPU (baseline/_ref), rank 0 only
    python bench.py --steps K --dump-outputs DIR                  # also write what the last timed step computed, as .npy

A "step" is one full training step of the MAGVIT2 VideoTokenizer (GAN / perceptual terms disabled — the
only configuration in which the reference runs offline, SURVEY.md §8) on one synthetic batch of
B x 3 x 16 x 64 x 64 video per GPU: forward, backward, (gradient all-reduce for N>1), fused AdamW.
One JSON line is printed by rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FRAMES, RES = 16, 64
# algorithmic conv FLOPs of one MAGVIT2 training step per clip (SURVEY.md §8d: 2506.1 GF forward, x3 for train)
CONV_GFLOP_FWD_PER_CLIP = 2506.1


def env_int(k, d):
    return int(os.environ.get(k, d))


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, 'measured (MEASURED_PEAKS.json)'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for ln in self.lines:
            parts = [x.strip() for x in ln.split(',')]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = float(parts[1])
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(nm)
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx, 'reasons': sorted(reasons),
                'samples': len(sm)}


# --------------------------------------------------------------------------------------------------
# CPU leg: the reference's OWN implementation (the unmodified myscience/open-genie package vendored by
# __graft_entry__.build() into baseline/_ref, imported through the `lightning` stand-in of oracle/_shim) on the
# host cores; if that copy is absent, the oracle port of the same algorithm (oracle/genie_oracle.py). A measured
# baseline only — never on the product path.
# --------------------------------------------------------------------------------------------------
REF_DIR = os.path.join(ROOT, 'baseline', '_ref')


def usable_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def pick_cpu_threads():
    """Thread policy of the CPU arm, stated in the JSON line: a FIXED min(32, usable cores) threads (OG_CPU_THREADS
    overrides). Measured on this pool's 128-thread hosts with the whole reference training step: 32 threads 1.99-2.27
    frames/s, 64 threads 1.32 frames/s (profiles/r02bb_*), and with all 128 threads a conv3d probe is 25-50x slower
    (oversubscription) — so `os.cpu_count()` threads would flatter the GPU/CPU ratio. Earlier rounds PICKED the count with
    a conv3d probe; the probe put 32 and 64 within 5 % of each other and flipped between runs, so it is now reported
    only (`thread_probe_ms`, conv3d forward+backward, best of 3) and no longer decides."""
    import torch.nn.functional as F
    avail = usable_cores()
    cands = sorted({c for c in (8, 16, 32, 64, avail) if c <= avail})
    x = torch.randn(1, 128, 8, 64, 64, requires_grad=True)
    w = torch.randn(128, 128, 3, 3, 3, requires_grad=True)
    probe = {}
    for c in cands:
        torch.set_num_threads(c)
        F.conv3d(x, w, padding=1).sum().backward()
        best = float('inf')
        for _ in range(3):
            t0 = time.perf_counter()
            F.conv3d(x, w, padding=1).sum().backward()
            best = min(best, time.perf_counter() - t0)
        probe[c] = round(best * 1e3, 1)
    env = os.environ.get('OG_CPU_THREADS')
    pick = max(1, min(int(env), avail)) if env else min(32, avail)
    torch.set_num_threads(pick)
    return pick, avail, probe


def cpu_train_step_factory(batch, seed=0):
    """One MAGVIT2 VideoTokenizer training step (fwd + bwd + AdamW, fp32) on `batch` clips. Returns (step, kind)."""
    torch.manual_seed(seed)
    video = torch.randn(batch, 3, FRAMES, RES, RES)
    if os.path.isdir(os.path.join(REF_DIR, 'genie')):
        for pth in (os.path.join(ROOT, 'oracle', '_shim'), REF_DIR):
            if pth not in sys.path:
                sys.path.insert(0, pth)
        import copy
        import torch.nn as nn
        from genie.tokenizer import MAGVIT2_DEC_DESC, MAGVIT2_ENC_DESC, VideoTokenizer   # the reference itself

        class ZeroLoss(nn.Module):          # GAN / perceptual terms off (VGG weights need a download): SURVEY.md §8c
            def forward(self, *a, **k):
                return torch.zeros(())

        model = VideoTokenizer(copy.deepcopy(MAGVIT2_ENC_DESC), copy.deepcopy(MAGVIT2_DEC_DESC), d_codebook=18,
                               gan_loss_weight=0, perc_loss_weight=0)
        model.gan_crit = model.perc_crit = ZeroLoss()
        model.train()
        opt = model.configure_optimizers()                  # the reference's default: torch.optim.AdamW

        def step():
            loss = model.training_step(video, 0)
            loss.backward()
            opt.step()
            opt.zero_grad(set_to_none=True)
            return float(loss.detach())
        return step, 'reference'
    from oracle import genie_oracle as O
    import open_genie_b200 as og
    model = og.VideoTokenizer(og.MAGVIT2_ENC_DESC, og.MAGVIT2_DEC_DESC, d_codebook=18, gan_loss_weight=0,
                              perc_loss_weight=0)          # CPU construction only: parameter shapes + default init
    sd = {k: v.detach().clone().contiguous().requires_grad_(v.dtype.is_floating_point)
          for k, v in model.state_dict().items()}
    params = [v for v in sd.values() if v.requires_grad]
    opt = torch.optim.AdamW(params)                         # the reference's default (genie/tokenizer.py:250)
    del model

    def step():
        loss, _, _, _ = O.tokenizer_forward(sd, og.MAGVIT2_ENC_DESC, og.MAGVIT2_DEC_DESC, video, 18)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return float(loss.detach())
    return step, 'port'


WORKLOAD = ('BASELINE configs[1]: MAGVIT2_ENC/DEC VideoTokenizer training step (fwd + bwd + AdamW), d_codebook=18, '
            f'{FRAMES}x{RES}x{RES} synthetic video, GAN+perceptual terms off (the reference runs offline only that way)')


def cpu_sample_text(batch, threads, avail, kind):
    what = ('unmodified reference package (baseline/_ref) through its own VideoTokenizer.training_step + AdamW'
            if kind == 'reference' else 'oracle/genie_oracle.py port of the reference (pinned to reference outputs)')
    return (f'{batch} clip(s) x {FRAMES} frames per step, fp32 torch CPU, {threads} threads (fixed policy min(32, cores): '
            f'the fastest count for this step on the {avail}-thread hosts, 64 threads measured 1.5x slower); {what}')


def run_reference(args, rank, world):
    if rank != 0:
        return
    threads, avail, probe = pick_cpu_threads()
    batch = args.cpu_batch
    step, kind = cpu_train_step_factory(batch)
    t0 = time.perf_counter()
    step()                                                  # first (untimed) step doubles as the time probe
    first = time.perf_counter() - t0
    if batch > 1 and first * (args.steps + args.warmup) > args.cpu_budget_s:
        batch = 1                                           # keep the whole run within a few minutes
        step, kind = cpu_train_step_factory(batch)
        step()
    for _ in range(max(args.warmup - 1, 0)):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / max(args.steps, 1)
    fps = batch * FRAMES / dt
    line = {
        'impl': 'reference', 'metric': 'videotokenizer_train_step_frames_per_sec', 'value': fps, 'unit': 'frames/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': WORKLOAD, 'cpu_sample_clips_per_step': batch},
        'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': threads, 'cores_usable': avail, 'kind': kind,
                         'thread_probe_ms': probe, 'sample': cpu_sample_text(batch, threads, avail, kind)},
        'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------------
# algorithmic HBM bytes of one launch of the bandwidth-bound kernels, from the C-ABI arguments (DESIGN.md §3:
# bf16 activations = 2 B/element; what each pass must read + write at minimum)
def _hbm_bytes(name, a):
    if name in ('og_gn_stats',):
        return 2.0 * a['N'] * a['V'] * a['C']
    if name in ('og_gn_act_fwd', 'og_affine_act_fwd'):
        return 4.0 * a['N'] * a['V'] * a['C']
    if name == 'og_affine_act_bwd_reduce':
        return 4.0 * a['N'] * a['V'] * a['C']
    if name in ('og_gn_act_bwd', 'og_affine_act_bwd_apply'):
        return (6.0 + (2.0 if a.get('add') else 0.0)) * a['N'] * a['V'] * a['C']
    if name == 'og_pixel_shuffle3d':
        return 4.0 * a['N'] * a['T'] * a['H'] * a['W'] * a['c'] * a['p'] * a['q'] * a['r']
    if name == 'og_colsum':
        return 2.0 * a['rows'] * a['C']
    if name == 'og_rope_ln_fwd':
        return 4.0 * a['rows'] * a['C']
    if name == 'og_ncdhw_f32_to_ndhwc':
        return (4.0 + (4.0 if a['y_f32'] else 2.0)) * a['N'] * a['C'] * a['V']
    if name in ('og_mse_fwd',):
        return 8.0 * a['N'] * a['C'] * a['V']
    if name == 'og_mse_bwd':
        return (8.0 * a['C'] + 2.0 * a['cpad']) * a['N'] * a['V']
    return None


DUMP_PER_PARAM = 4096      # values per parameter in params_sample.npy: 0.67 M of the 375 M parameters, 2.7 MB


def dump_outputs(out_dir, loss, model):
    """What the last timed step hands its caller: the loss, and the parameters the optimizer step left behind (a fixed,
    seeded sample of DUMP_PER_PARAM values of each, in named_parameters() order). Both float32."""
    import numpy as np
    gen = torch.Generator().manual_seed(0)
    parts = []
    for _, p in model.named_parameters():
        flat = p.detach().flatten()
        if flat.numel() > DUMP_PER_PARAM:
            flat = flat[torch.randint(flat.numel(), (DUMP_PER_PARAM,), generator=gen).to(flat.device)]
        parts.append(flat.float().cpu())
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, 'loss.npy'), loss.detach().float().cpu().reshape(1).numpy())
    np.save(os.path.join(out_dir, 'params_sample.npy'), torch.cat(parts).numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--batch', type=int, default=8, help='clips per GPU (BASELINE configs[1]: 8)')
    ap.add_argument('--cpu-batch', type=int, default=2, help='clips per CPU-baseline step (BASELINE.md §3: B = 2)')
    ap.add_argument('--cpu-budget-s', type=float, default=300.0,
                    help='--impl reference: drop to 1 clip per step if (steps+warmup) x first-step time exceeds this')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-graph', action='store_true', help='launch every kernel from Python instead of replaying the captured step')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the loss and a sample of the updated parameters of the last one')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    rank, world, local = env_int('RANK', 0), env_int('WORLD_SIZE', 1), env_int('LOCAL_RANK', 0)

    if args.impl == 'reference':
        run_reference(args, rank, world)
        return

    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # Every CTA NCCL occupies takes a whole SM away from the persistent one-CTA-per-SM GEMM kernels (227 KB of shared
        # memory each: nothing co-resides); capping NCCL's CTAs was measured and is WORSE (N = 2, profiles/r02j_*: 8 CTAs
        # 66.3 ms = default, 4 CTAs 69.7, 2 CTAs 81.3 — the all-reduce then no longer hides behind backward). The GEMM
        # kernels instead draw their tiles dynamically, so CTAs that cannot be resident cost nothing (conv3d_igemm.cu).
        if os.environ.get('OG_NCCL_MAX_CTAS'):
            os.environ.setdefault('NCCL_MAX_CTAS', os.environ['OG_NCCL_MAX_CTAS'])
        dist.init_process_group('nccl', device_id=dev)

    import open_genie_b200 as og
    from open_genie_b200 import _lib, ops
    from open_genie_b200.ddp import ArenaGradAllReducer

    torch.manual_seed(0)
    model = og.VideoTokenizer(og.MAGVIT2_ENC_DESC, og.MAGVIT2_DEC_DESC, d_codebook=18, gan_loss_weight=0,
                              perc_loss_weight=0).to(dev)
    n_params = sum(p.numel() for p in model.parameters())
    opt = model.configure_optimizers()                      # FusedAdamW, AdamW defaults
    og.enable_zero_arena(True)   # every step below ends with zero_grad(set_to_none=True): the arena contract holds
    # N > 1: ONE gradient exchange per step, all-reduced in place on the step's zero arena (no bucket copies)
    bucket_mb = int(os.environ.get('OG_BUCKET_MB', '64'))
    reducer = ArenaGradAllReducer(model.parameters(), bucket_bytes=bucket_mb << 20) if world > 1 else None
    if os.environ.get('OG_DDP_MODE') == 'none':     # diagnosis only: N independent replicas, no gradient exchange
        for h in reducer._hooks:
            h.remove()
        reducer = None
    B = args.batch
    torch.manual_seed(1234 + rank)
    host_video = torch.randn(B, 3, FRAMES, RES, RES).pin_memory()
    dev_video = host_video.to(dev)
    h2d_bytes = host_video.numel() * 4

    def eager_step(video):
        loss = model.training_step(video, 0)
        loss.backward()
        if reducer is not None:
            reducer.finish()
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------- warm-up (>= 3 steps) + capture of the whole step into one CUDA graph ----------------
    for _ in range(max(args.warmup, 3)):
        eager_step(dev_video)
    barrier()
    use_graph = not args.no_graph
    graph_note = None
    if use_graph:
        from open_genie_b200.graph import GraphedTrainStep
        ok = torch.ones(1, device=dev)
        try:
            train_step = GraphedTrainStep(model, opt, dev_video, warmup=3, reducer=reducer)
        except Exception as e:                              # every rank must take the same path
            graph_note = f'{type(e).__name__}: {e}'[:200]
            ok.zero_()
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if float(ok.item()) == 0.0:
            use_graph = False
            if reducer is not None:
                reducer.bind_arena(None)
            model.zero_grad(set_to_none=True)
    if use_graph:
        for _ in range(2):
            train_step(dev_video)
    else:
        train_step = eager_step
    barrier()

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            out = fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1)), out

    def e2e_step():
        if use_graph:
            loss = train_step(host_video)                  # H2D from pinned memory into the static input + replay
        else:
            loss = train_step(host_video.to(dev, non_blocking=True))
        _ = loss.item()                                    # D2H read of the step's result

    # ---------------- timed legs: e2e (a) -> device-resident `value` -> e2e (b) ----------------
    # The e2e leg brackets the value leg on both sides so that slow clock drift under the power cap cancels in the
    # comparison of the two (round 1 ran them back to back and e2e came out 1 % FASTER than value).
    ms_e2e_a, _ = timed(e2e_step)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.launch_count()
    ms_total, last_loss = timed(lambda: train_step(dev_video))
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs and rank == 0:      # before the next leg replays the step again
        dump_outputs(args.dump_outputs, last_loss, model)
    ms_e2e_b, _ = timed(e2e_step)
    ms_e2e = 0.5 * (ms_e2e_a + ms_e2e_b)

    # ---------------- per-kernel timing pass (eager, CUDA events around every launch of the library) ----------
    # A replayed graph cannot carry timing events, so the roofline numbers come from the same step launched
    # eagerly right after the timed region (same process, same inputs, same kernels and grid sizes).
    model.zero_grad(set_to_none=True)
    if reducer is not None:
        reducer.bind_arena(None)
    prof_steps = min(args.steps, 3)
    eager_step(dev_video)                                   # re-sizes the default scope's arena after the graph's private one
    ops.PROFILE = []
    _lib.TIMING = []
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    eager_launch0 = _lib.launch_count()
    p0.record()
    for _ in range(prof_steps):
        eager_step(dev_video)
    p1.record()
    barrier()
    ms_prof = p0.elapsed_time(p1)
    launches_per_step = (_lib.launch_count() - eager_launch0) / prof_steps
    prof, ops.PROFILE = ops.PROFILE, None
    timing, _lib.TIMING = _lib.TIMING, None
    if use_graph:
        launches = int(round(launches_per_step * args.steps))   # kernels executed by the replays of the timed region

    if rank == 0:
        peaks, peak_src = load_peaks()
        ms_step = ms_total / args.steps
        fps = world * B * FRAMES / (ms_step * 1e-3)
        fps_e2e = world * B * FRAMES / (ms_e2e / args.steps * 1e-3)
        # per-kernel roofline from the CUDA events recorded around every tensor-core launch
        kinds = {}
        for kind, flops, a, b, _shape in prof:
            k = 'og_conv_wgrad_kernel' if kind == 'wgrad' else 'og_conv_igemm_kernel'
            d = kinds.setdefault(k, {'ms': 0.0, 'flop': 0.0, 'launches': 0})
            d['ms'] += a.elapsed_time(b)
            d['flop'] += flops
            d['launches'] += 1
        peak_tf = peaks.get('bf16_tflops_sustained', peaks.get('bf16_tflops'))
        peak_bw = peaks.get('hbm_gbs')
        # the ten conv problem shapes that cost the most time per step (small-int C-ABI arguments identify the layer)
        by_shape = {}
        for kind, flops, a, b, shape in prof:
            d = by_shape.setdefault((kind,) + tuple(shape), {'ms': 0.0, 'flop': 0.0, 'n': 0})
            d['ms'] += a.elapsed_time(b)
            d['flop'] += flops
            d['n'] += 1
        top_shapes = [{'kind': k[0], 'args': list(k[1:]), 'launches_per_step': d['n'] / prof_steps,
                       'ms_per_step': round(d['ms'] / prof_steps, 3), 'tflops': round(d['flop'] / max(d['ms'], 1e-9) * 1e-9, 1)}
                      for k, d in sorted(by_shape.items(), key=lambda kv: -kv[1]['ms'])[:14]]
        kern = {}
        for k, d in kinds.items():
            tf = d['flop'] / max(d['ms'], 1e-9) * 1e-9
            kern[k] = {'bound': 'tensor', 'launches_per_step': d['launches'] / prof_steps, 'ms_per_step': d['ms'] / prof_steps,
                       'tflops': tf, 'frac': tf / peak_tf, 'share_of_step': (d['ms'] / prof_steps) / max(ms_step, 1e-9)}
        # HBM-bound passes: algorithmic bytes (from the C-ABI arguments) / event time, against the measured copy bandwidth
        hb = {}
        for name, cargs, a, b in timing:
            if name.startswith('og_conv3d'):
                continue
            named = dict(zip(_lib.PROTOTYPES[name][2], cargs))
            d = hb.setdefault(name, {'ms': 0.0, 'bytes': 0.0, 'launches': 0, 'known': True, 'ms_big': 0.0, 'bytes_big': 0.0,
                                     'n_big': 0})
            dt = a.elapsed_time(b)
            d['ms'] += dt
            d['launches'] += 1
            nb = _hbm_bytes(name, named)
            if nb is None:
                d['known'] = False
            else:
                d['bytes'] += nb
                if nb >= 32e6:      # launches large enough that the eager launch gap (~10 us of CPU per call) is not what the
                    d['ms_big'] += dt   # events measure: these show the kernel, the aggregate shows the step
                    d['bytes_big'] += nb
                    d['n_big'] += 1
        if 'og_adamw_step' in hb:        # 4 fp32 reads (p, g, m, v) + 3 fp32 writes + the bf16 operand copy of conv weights
            hb['og_adamw_step']['bytes'] = 30.0 * n_params * prof_steps
            hb['og_adamw_step']['known'] = True
        for name, d in hb.items():
            e = {'bound': 'hbm', 'launches_per_step': d['launches'] / prof_steps, 'ms_per_step': d['ms'] / prof_steps,
                 'share_of_step': (d['ms'] / prof_steps) / max(ms_step, 1e-9)}
            if d['known'] and d['bytes'] > 0:
                gbs = d['bytes'] / max(d['ms'], 1e-9) * 1e-6
                e.update(gbs=gbs, frac=gbs / peak_bw)
                if d['n_big']:
                    gb = d['bytes_big'] / max(d['ms_big'], 1e-9) * 1e-6
                    e.update(large_launches={'count_per_step': d['n_big'] / prof_steps, 'gbs': gb, 'frac': gb / peak_bw,
                                             'min_algorithmic_bytes': 32e6})
            kern[name] = e
        dom = max(kinds, key=lambda k: kern[k]['ms_per_step']) if kinds else None
        roofline = None
        if dom:
            traffic, traffic_note = None, None
            try:    # DRAM bytes of one launch of the dominant kernel, from the committed ncu --set full capture
                tj = json.load(open(os.path.join(ROOT, 'profiles', 'r02_ncu_traffic.json')))[dom]
                traffic = tj['traffic_bytes']
                traffic_note = (f"ncu --set full, one launch of {tj['shape']}: dram read {tj['dram_read_bytes']} + "
                                f"write {tj['dram_write_bytes']} B; algorithmic {tj['algorithmic_bytes']} B")
            except Exception:
                pass
            conv_flop = sum(d['flop'] for d in kinds.values()) / prof_steps
            roofline = {'kernel': dom, 'bound': 'tensor', 'achieved': kern[dom]['tflops'], 'peak': peak_tf,
                        'unit': 'TFLOP/s', 'frac': kern[dom]['tflops'] / peak_tf, 'traffic': traffic,
                        'traffic_note': traffic_note,
                        'peak_source': peak_src + ' sustained bf16; HBM-bound kernels against hbm_gbs', 'kernels': kern,
                        'conv_flop_per_step': conv_flop, 'conv_top_shapes': top_shapes,
                        'whole_step': {'tflops': conv_flop / (ms_step * 1e-3) * 1e-12,
                                       'frac': conv_flop / (ms_step * 1e-3) * 1e-12 / peak_tf},
                        'timing': f'CUDA events around each launch over {prof_steps} eagerly launched steps after the '
                                  f'timed region ({ms_prof / prof_steps:.1f} ms/step eager)'}
        launch = 'whole step (fwd + bwd + NCCL all-reduce + AdamW) replayed as one CUDA graph' if use_graph else \
            'eager launches' + (f' (graph capture failed: {graph_note})' if graph_note else '')
        line = {
            'metric': 'videotokenizer_train_step_frames_per_sec', 'value': fps, 'unit': 'frames/s', 'n_gpus': world,
            'steps': args.steps, 'warmup': max(args.warmup, 3), 'ms_per_step': ms_step, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
            'config': {'workload': WORKLOAD + '; bf16 compute / fp32 master weights',
                       'batch_per_gpu': B, 'global_batch': B * world, 'frames': FRAMES, 'resolution': RES,
                       'params': n_params, 'parallelism': f'dp{world}', 'launch': launch,
                       'grad_exchange': None if reducer is None else
                       f'NCCL all-reduce (AVG) in place on the zero arena, {reducer.bucket >> 20} MB ranges overlapped with '
                       f'backward, {reducer.grad_bytes()} B per step, NCCL_MAX_CTAS={os.environ.get("NCCL_MAX_CTAS")}',
                       'l2': 'no flush: every step streams several GB of activations (>> 126 MB L2)'},
            'e2e': {'value': fps_e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': h2d_bytes * world,
                    'd2h_bytes_per_step': 4 * world,
                    'legs_ms': [ms_e2e_a / args.steps, ms_e2e_b / args.steps],
                    'note': 'mean of two K-step legs bracketing the device-resident leg'},
            'gpu_launches': int(launches),
            'clocks': clocks,
            'roofline': roofline,
        }
        if world == 1 and not args.no_cpu_baseline:
            threads, avail, probe = pick_cpu_threads()
            step, kind = cpu_train_step_factory(args.cpu_batch)
            t0 = time.perf_counter()
            step()
            dt = time.perf_counter() - t0
            line['cpu_baseline'] = {
                'value': args.cpu_batch * FRAMES / dt, 'unit': 'frames/s', 'cores': threads, 'cores_usable': avail,
                'kind': kind, 'thread_probe_ms': probe,
                'sample': f'one training step ({dt:.1f} s): ' + cpu_sample_text(args.cpu_batch, threads, avail, kind)}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tearing the process group down while a CUDA graph that captured NCCL collectives is still alive hung in
        # ProcessGroupNCCL's destructor (2xB200, torch 2.11 / NCCL 2.28): finish all work, agree that everybody is done,
        # then leave without running the destructors.
        barrier()
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


if __name__ == '__main__':
    main()
