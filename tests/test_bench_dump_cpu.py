"""bench.py --dump-outputs on the CPU: what dump_outputs writes for a padded detection payload (no kernel is called)."""
import os

import numpy as np
import torch

import bench
from gencomm_b200 import shard


def _payload():
    g = torch.Generator().manual_seed(3)
    boxes, scores = torch.randn(4, 1000, 8, 3, generator=g), torch.rand(4, 1000, generator=g)
    counts = torch.tensor([0, 5, 1000, 17], dtype=torch.int32)
    return boxes, scores, counts, shard.pack_detections(boxes, scores, counts)


def test_dump_outputs_writes_the_detections_with_padding_zeroed(tmp_path):
    boxes, scores, counts, payload = _payload()
    bench.dump_outputs(str(tmp_path), payload)
    d = {n[:-4]: np.load(tmp_path / n) for n in os.listdir(tmp_path)}
    assert sorted(d) == ["boxes", "counts", "frames", "scores"]
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert d["frames"].tolist() == [0, 1, 2, 3] and d["counts"].tolist() == [0, 5, 1000, 17]
    assert d["boxes"].shape == (4, 1000, 8, 3) and d["scores"].shape == (4, 1000)
    for f, k in enumerate(counts.tolist()):
        assert np.array_equal(d["boxes"][f, :k], boxes[f, :k].numpy()) and not d["boxes"][f, k:].any()
        assert np.array_equal(d["scores"][f, :k], scores[f, :k].numpy()) and not d["scores"][f, k:].any()


def test_dump_outputs_samples_frames_above_the_size_limit(tmp_path, monkeypatch):
    boxes, _, counts, payload = _payload()
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 2 * (shard.DET_WIDTH * 4 + 8))
    bench.dump_outputs(str(tmp_path / "a"), payload)
    bench.dump_outputs(str(tmp_path / "b"), payload)
    total = sum(os.path.getsize(tmp_path / "a" / n) for n in os.listdir(tmp_path / "a"))
    frames = np.load(tmp_path / "a" / "frames.npy").astype(int)
    assert len(frames) == 2 and total <= bench.DUMP_LIMIT_BYTES + 4 * 128          # + the .npy headers
    assert np.array_equal(frames, np.load(tmp_path / "b" / "frames.npy"))           # the same sample every run
    assert np.load(tmp_path / "a" / "counts.npy").tolist() == counts[frames].tolist()
    f = frames[-1]
    k = int(counts[f])
    assert np.array_equal(np.load(tmp_path / "a" / "boxes.npy")[-1, :k], boxes[f, :k].numpy())
