"""Host-side logic that needs no GPU: API surface, state_dict layout, sharding (gloo, world 2)."""
import os
import socket

import numpy as np
import pytest
import torch

import pixeltable_yolox_b200 as yx
from pixeltable_yolox_b200.sharding import shard_range


def test_named_configs_and_param_counts():
    # docs/model_zoo.md:7-10,30-31 (params in M)
    want = {"yolox_nano": 0.91, "yolox_tiny": 5.06, "yolox_s": 8.97, "yolox_m": 25.33, "yolox_l": 54.21, "yolox_x": 99.07}
    for name, m_params in want.items():
        cfg = yx.YoloxConfig.get_named_config(name)
        cfg.model = None
        model = cfg.get_model()
        n = sum(p.numel() for p in model.parameters()) / 1e6
        assert abs(n - m_params) < 0.02, (name, n)
        assert model.training          # get_model() returns train mode (config.py:176)
        cfg.model = None
    assert yx.YoloxConfig.get_named_config("yolox-s") is yx.YoloxConfig.get_named_config("yolox_s")
    assert yx.YoloxConfig.get_named_config("nope") is None


def test_get_model_is_cached_on_the_config_like_the_reference():
    cfg = yx.YoloxConfig("c", depth=0.33, width=0.25)
    assert cfg.get_model() is cfg.get_model()
    b = cfg.get_model().head.cls_preds[0].bias
    assert torch.allclose(b, torch.full_like(b, -np.log(99.0)))


def test_eval_on_cpu_raises_instead_of_falling_back():
    cfg = yx.YoloxConfig("c", depth=0.33, width=0.25)
    m = cfg.get_model().eval()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        m(torch.zeros(1, 3, 64, 64))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        yx.postprocess(torch.zeros(1, 10, 85), 80)
    with pytest.raises(IndexError):
        yx.bboxes_iou(torch.zeros(2, 3), torch.zeros(2, 4))
    with pytest.raises(AssertionError):
        cfg.get_model().train()(torch.zeros(1, 3, 64, 64))     # training without targets (yolox.py:77)


def test_from_pretrained_errors_match_reference():
    with pytest.raises(ValueError, match="Unknown model"):
        yx.YoloxModule.from_pretrained("not_a_model")
    with pytest.raises(ValueError):
        yx.YoloxProcessor(3)


def test_processor_letterbox_matches_reference_preproc():
    from PIL import Image

    rng = np.random.default_rng(0)
    img = Image.fromarray(rng.integers(0, 255, size=(48, 64, 3), dtype=np.uint8))
    proc = yx.YoloxProcessor("yolox_nano")
    t = proc([img])
    assert t.shape == (1, 3, 416, 416) and t.dtype == torch.float32
    r = min(416 / 48, 416 / 64)
    assert (t[0, :, int(48 * r):, :] == 114).all()        # grey padding below the resized image
    assert t.max() <= 255 and t.min() >= 0 and (t == t.floor()).all()


def test_shard_range_partitions():
    for n in (0, 1, 7, 64, 513):
        for world in (1, 2, 3, 8):
            spans = [shard_range(n, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [e - b for b, e in spans]
            assert max(sizes) - min(sizes) <= 1


def _worker(rank, world, port, q):
    import torch.distributed as dist

    from pixeltable_yolox_b200.sharding import gather_detection_counts, shard_range

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    b, e = shard_range(13, rank, world)
    counts = gather_detection_counts([i * i for i in range(b, e)])
    # the path has no data-path collective; the only traffic is this metadata gather
    t = torch.tensor([e - b], dtype=torch.int64)
    dist.all_reduce(t)
    q.put((rank, counts, int(t.item())))
    dist.destroy_process_group()


def test_two_rank_batch_sharding_gloo():
    import torch.multiprocessing as mp

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=120) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    for rank, counts, total in res:
        assert counts == [i * i for i in range(13)] and total == 13


def test_set_match_comparator():
    """The IoU >= 0.99 one-to-one comparator of the north_star gate (used by tests/test_gpu_named_configs.py)."""
    from test_gpu_named_configs import match_sets

    a = np.array([[10, 10, 110, 110, .9, .9, 3], [200, 200, 300, 320, .8, .9, 5], [10, 10, 110, 110, .7, .9, 4]], dtype=np.float32)
    b = a.copy()
    assert match_sets([a], [b]) == 3
    b[0, :4] += 0.2                          # IoU ~0.992: still a match; 2 px shift is not
    assert match_sets([a], [b]) == 3
    b[1, :4] += 2.0
    assert match_sets([a], [b]) == 2
    b[2, 6] = 7                              # label differs
    assert match_sets([a], [b]) == 1
    assert match_sets([a, None], [b, a]) == 1 and match_sets([a], [None]) == 0
    assert match_sets([a], [np.concatenate([a, a])]) == 3          # one-to-one: duplicates do not count twice


def test_bench_dump_outputs(tmp_path):
    """bench.py --dump-outputs on an engine's output buffers: float32 / float64 arrays within 64 MB, the detections of each
    image up to its kept count (at most max_det) and cleared after it, the same seeded sample of head-output rows every run."""
    import types

    import bench

    B, A, nc, max_det = 8, 8400, 80, 1000
    g = torch.Generator().manual_seed(0)
    eng = types.SimpleNamespace(det_count=torch.randint(0, 50, (B,), dtype=torch.int32, generator=g),
                                dets=torch.randn(B, max_det, 7, generator=g),
                                det_idx=torch.randint(0, B * A, (B, max_det), generator=g),
                                pred=torch.randn(B, A, 5 + nc, generator=g))
    eng.det_count[1] = max_det + 5
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), eng, max_det)
    files = sorted(p.name for p in (tmp_path / "a").iterdir())
    assert files == ["det_count.npy", "det_idx.npy", "dets.npy", "pred_rows.npy", "pred_rows_index.npy"]
    assert sum((tmp_path / "a" / f).stat().st_size for f in files) <= 64 << 20
    out = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert out[f[:-4]].dtype in (np.float32, np.float64)
        assert np.array_equal(out[f[:-4]], np.load(tmp_path / "b" / f))
    np.testing.assert_array_equal(out["det_count"], eng.det_count.numpy())
    kept = np.minimum(eng.det_count.numpy(), max_det)
    assert out["dets"].shape == (B, max_det, 7) and out["det_idx"].shape == (B, max_det)
    for b, k in enumerate(kept):
        np.testing.assert_array_equal(out["dets"][b, :k], eng.dets[b, :k].numpy())
        np.testing.assert_array_equal(out["det_idx"][b, :k], eng.det_idx[b, :k].numpy())
        assert (out["dets"][b, k:] == 0).all() and (out["det_idx"][b, k:] == -1).all()
    rows = out["pred_rows_index"].astype(np.int64)
    assert len(rows) == bench.PRED_SAMPLE_ROWS < B * A and len(np.unique(rows)) == len(rows)
    np.testing.assert_array_equal(out["pred_rows"], eng.pred.reshape(B * A, 5 + nc)[rows].numpy())
