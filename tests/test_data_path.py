"""Data path (SURVEY.md §8 f4): Platformer2D / LightningPlatformer2D on mp4 files written here with OpenCV (CPU),
against what the reference's own Platformer2D returned for the same files (tests/golden/platformer.pt, written by
oracle/make_golden.py), and the device-side frame decode + prefetcher (GPU)."""
import os

import pytest
import torch

from oracle import fixtures as fx
from oracle import genie_oracle as O


@pytest.fixture(scope='module')
def clips(tmp_path_factory):
    pytest.importorskip('cv2')
    root = tmp_path_factory.mktemp('platformer')
    fx.write_platformer_clips(str(root))
    return str(root)


def test_platformer2d_matches_the_reference_dataset(clips, golden):
    import open_genie_b200 as og
    ref = golden('platformer.pt')
    for fmt in ('t c h w', 'c t h w'):
        for padding in ('none', 'repeat', 'zero'):
            ds = og.Platformer2D(clips, split='train', padding=padding, num_frames=16, output_format=fmt)
            assert len(ds) == 5
            v = ds[1]
            shape = (16, 3, 64, 64) if fmt == 't c h w' else (3, 16, 64, 64)
            assert v.shape == shape and v.dtype == torch.float32 and 0.0 <= float(v.min()) and float(v.max()) <= 1.0
            short = [ds[i] for i in range(5) if ds.file_names[i].endswith('clip0.mp4')][0]
            assert short.shape[0 if fmt == 't c h w' else 1] == 12        # whole (shorter) video: data.py:191-193
            root = os.path.join(clips, 'Coinrun', 'train')
            assert ds.file_names == [os.path.join(root, f) for f in os.listdir(root)]     # data.py:163-166
            for i, f in enumerate(ds.file_names):
                key = (fmt, padding, os.path.basename(f))
                want = ref[key]['x255'].float() / 255.                                 # exactly the reference's values
                assert tuple(ds[i].shape) == ref[key]['shape']
                assert torch.equal(O.det_sample(ds[i], 'platformer.{}.{}.{}'.format(*key), want.numel()), want)
    raw = og.Platformer2D(clips, split='val', num_frames=16, raw_uint8=True)[0]
    assert raw.dtype == torch.uint8 and raw.shape == (16, 64, 64, 3)
    ref = og.Platformer2D(clips, split='val', num_frames=16, output_format='t h w c')[0]
    assert torch.equal(raw.flip(-1).float() / 255., ref)                       # raw frames are BGR


def test_lightning_datamodule_surface(clips, tmp_path):
    import open_genie_b200 as og
    dm = og.LightningPlatformer2D(clips, num_frames=16, output_format='c t h w', batch_size=2, num_workers=0)
    dm.setup('fit')
    batch = next(iter(dm.train_dataloader()))
    assert batch.shape[0] == 2 and batch.shape[1] == 3 and batch.dtype == torch.float32
    assert len(dm.valid_dataset) == 2
    dm.setup('test')
    assert len(dm.test__dataset) == 2
    with pytest.raises(ValueError, match='Invalid stage'):
        dm.setup('nope')
    with pytest.raises(NotImplementedError):
        og.LightningDataset().setup('fit')
    cfg = tmp_path / 'conf.yaml'
    cfg.write_text(f'dataset:\n  root: {clips}\n  num_frames: 8\n  batch_size: 3\n')
    dm2 = og.LightningPlatformer2D.from_config(str(cfg))
    assert dm2.num_frames == 8 and dm2.batch_size == 3


@pytest.mark.gpu
def test_device_frame_decode_and_prefetcher(clips):
    import open_genie_b200 as og
    from open_genie_b200 import ops
    torch.manual_seed(0)
    frames = torch.randint(0, 256, (2, 4, 16, 16, 3), dtype=torch.uint8)
    want = (frames.flip(-1).float() / 255.).permute(0, 4, 1, 2, 3).contiguous()      # BGR -> RGB, /255, 'c t h w'
    got = og.frames_to_video(frames.cuda())
    assert got.shape == (2, 3, 4, 16, 16) and torch.equal(got.cpu(), want)            # exact: same fp32 arithmetic
    gi = og.frames_to_video(frames.cuda(), internal=True, cpad=8)
    assert ops.is_internal(gi[:, :3].contiguous(memory_format=torch.channels_last_3d)) or gi.shape == (2, 3, 4, 16, 16)
    assert torch.equal(gi.float().cpu(), want.to(torch.bfloat16).float())
    # end to end: uint8 loader -> pinned staging -> side-stream copy + decode == the reference-format CPU pipeline
    ds_raw = og.Platformer2D(clips, split='test', num_frames=16, raw_uint8=True)
    ds_ref = og.Platformer2D(clips, split='test', num_frames=16, output_format='c t h w')
    loader = torch.utils.data.DataLoader(ds_raw, batch_size=1, shuffle=False)
    pf = og.VideoBatchPrefetcher(loader)
    seen, elems = 0, 0
    for i, video in enumerate(pf):
        assert video.is_cuda and torch.equal(video[0].cpu(), ds_ref[i])
        seen += 1
        elems += video.numel()
    assert seen == len(ds_raw) and pf.h2d_bytes == elems                                # 1 byte per element over PCIe
