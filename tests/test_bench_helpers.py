"""Host-side helpers of bench.py that do not need a GPU: the static ncu traffic figure the `roofline` object quotes
and the algorithmic work table it is compared with (SURVEY 8d: 385.406 GFLOP, ~609 MB per image at 512 x 512)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def test_ncu_traffic_covers_every_launch_of_the_shipped_plan():
    """The newest committed `ncu --set full` capture must describe the 18-launch plan and every kernel family in it
    must be recognised (a renamed kernel once dropped two launches and the figure silently became null)."""
    import bench
    traffic, src = bench.ncu_traffic_bytes(18)
    assert traffic is not None and src.endswith("_ncu_raw.csv"), (traffic, src)
    # 17 non-stem launches of a batch-64 step: algorithmic 28.7 GB; a capture far off means mislabelled rows
    assert 24e9 < traffic < 34e9, traffic
    assert bench.ncu_traffic_bytes(22) == (None, None)          # another plan's launch count is refused


def test_dump_outputs_whole_images_seeded_sample_under_cap(tmp_path, monkeypatch):
    """--dump-outputs writes float32 whole images: every image when they fit the cap, else the same seeded sample of
    batch positions for each output, and never more than the cap in all."""
    import numpy as np
    import torch
    import bench
    g = torch.Generator().manual_seed(0)
    logits = torch.randn((64, 3, 16, 16), generator=g)
    mask = (logits > 0).to(torch.uint8)
    per_image = 2 * 3 * 16 * 16 * 4
    idx = bench.dump_outputs(str(tmp_path / "all"), {"logits": logits, "mask": mask})
    assert list(idx) == list(range(64))
    monkeypatch.setattr(bench, "DUMP_BYTES", 10 * per_image + 1024)
    dumps = [bench.dump_outputs(str(tmp_path / d), {"logits": logits, "mask": mask}) for d in ("a", "b")]
    assert np.array_equal(dumps[0], dumps[1]) and len(dumps[0]) == 10 and list(dumps[0]) == sorted(set(dumps[0]))
    for d, full in (("all", None), ("a", dumps[0])):
        files = sorted(os.listdir(tmp_path / d))
        assert files == ["image_index.npy", "logits.npy", "mask.npy"]
        if full is not None:
            assert sum(os.path.getsize(tmp_path / d / f) for f in files) <= bench.DUMP_BYTES
        keep = np.load(tmp_path / d / "image_index.npy").astype(np.int64)
        z, m = np.load(tmp_path / d / "logits.npy"), np.load(tmp_path / d / "mask.npy")
        assert z.dtype == m.dtype == np.float32
        assert np.array_equal(z, logits.numpy()[keep]) and np.array_equal(m, mask.numpy()[keep].astype(np.float32))


def test_bench_refuses_zero_timed_steps():
    import subprocess
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True)
    assert res.returncode == 2 and "--steps" in res.stderr
