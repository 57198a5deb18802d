"""bench.py --dump-outputs: what the last timed step computed, in the caller's logical layouts,
within the byte budget, sampled at the same seeded positions every run."""
import types

import numpy as np
import torch

import bench
from mvsdet_b200.scene import tiny_config


def _fake_pipe(cfg, seed):
    """The output buffers of a ScenePipeline, in its memory layouts, on the CPU."""
    v, c, d, t = cfg.n_views, cfg.channels, cfg.num_depth, cfg.topk
    hf, wf = cfg.feat_hw
    n = cfg.n_voxels[0] * cfg.n_voxels[1] * cfg.n_voxels[2]
    g = torch.Generator().manual_seed(seed)
    return types.SimpleNamespace(
        cfg=cfg, variance=torch.randn(v, d, hf, wf, c, generator=g),
        prob_volume=torch.rand(v, d, hf, wf, generator=g), off_pred=torch.rand(v, d, hf, wf, generator=g),
        est_depth=torch.rand(v, t, hf, wf, generator=g), est_dens=torch.rand(v, t, hf, wf, generator=g),
        est_idx=torch.randint(0, d, (v, t, hf, wf), generator=g),
        depth_coding=torch.rand(v, hf, wf, generator=g), volume_mean=torch.randn(c, n, generator=g),
        count=torch.randint(0, v, (n,), dtype=torch.int32, generator=g),
        g_feature=torch.randn(v, c, hf, wf, generator=g), g_cost_out=torch.randn(v, 2, d, hf, wf, generator=g))


def test_dump_is_logical_layout_within_budget_and_reproducible(monkeypatch, tmp_path):
    cfg = tiny_config()
    monkeypatch.setattr(bench, "DUMP_BUDGET", 11 * 4 * 2000)          # 2000 elements per output
    pipe = _fake_pipe(cfg, 0)
    arrays, info = bench.snapshot_outputs(pipe)
    assert sum(a.nbytes for a in arrays.values()) <= bench.DUMP_BUDGET
    assert all(a.dtype == np.float32 for a in arrays.values())
    # small outputs whole, in their logical shapes
    assert np.array_equal(arrays["count"], pipe.count.view(*cfg.n_voxels).float().numpy())
    assert np.array_equal(arrays["depth_coding"], pipe.depth_coding.numpy())
    # large ones sampled at seeded positions of the logical [V,C,D,Hf,Wf] index
    assert info["variance"]["sampled"] == arrays["variance"].size == 2000
    logical = pipe.variance.permute(0, 4, 1, 2, 3).reshape(-1).numpy()
    flat = np.sort(np.random.default_rng(0).choice(logical.size, 2000, replace=False))
    assert np.array_equal(arrays["variance"], logical[flat])
    # another run picks the same positions; other values give other samples
    again, _ = bench.snapshot_outputs(pipe)
    other, _ = bench.snapshot_outputs(_fake_pipe(cfg, 1))
    assert all(np.array_equal(arrays[k], again[k]) for k in arrays)
    assert not np.array_equal(arrays["g_feature"], other["g_feature"])
    bench.write_outputs(str(tmp_path / "out"), arrays)
    assert sorted(p.name for p in (tmp_path / "out").iterdir()) == sorted(f"{k}.npy" for k in arrays)
    assert np.array_equal(np.load(tmp_path / "out" / "volume_mean.npy"), arrays["volume_mean"])
