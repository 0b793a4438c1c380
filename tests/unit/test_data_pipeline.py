import numpy as np
import pytest
import torch
from torch import nn


def test_curriculum_schedules():
    from deepspeed_b200.runtime.data_pipeline.curriculum_scheduler import CurriculumScheduler
    s = CurriculumScheduler({"min_difficulty": 8, "max_difficulty": 64, "schedule_type": "fixed_linear",
                             "schedule_config": {"total_curriculum_step": 100, "difficulty_step": 8}})
    assert s.update_difficulty(0) == 8 and s.update_difficulty(50) == 32 and s.update_difficulty(100) == 64
    assert s.update_difficulty(1000) == 64
    r = CurriculumScheduler({"min_difficulty": 8, "max_difficulty": 64, "schedule_type": "fixed_root",
                             "schedule_config": {"total_curriculum_step": 100, "difficulty_step": 8, "root_degree": 2}})
    assert r.get_difficulty(25) == 32  # sqrt(0.25) = 0.5 -> 8 + 28 = 36 -> floor to 32
    d = CurriculumScheduler({"min_difficulty": 1, "max_difficulty": 3, "schedule_type": "fixed_discrete",
                             "schedule_config": {"difficulty": [1, 2, 3], "max_step": [5, 10]}})
    assert [d.get_difficulty(i) for i in (1, 5, 6, 10, 11)] == [1, 1, 2, 2, 3]
    c = CurriculumScheduler({"min_difficulty": 1, "max_difficulty": 9, "schedule_type": "custom"})
    c.set_custom_get_difficulty(lambda step: min(9, step))
    assert c.update_difficulty(4) == 4


def test_indexed_dataset_analyzer_sampler(tmp_path):
    from deepspeed_b200.runtime.data_pipeline.data_sampling import (DataAnalyzer, DeepSpeedDataSampler, MMapIndexedDataset,
                                                                   MMapIndexedDatasetBuilder)
    b = MMapIndexedDatasetBuilder(str(tmp_path / "d.bin"), dtype=np.int32)
    rows = [np.arange(n, dtype=np.int32) for n in (3, 5, 1, 4)]
    for r in rows:
        b.add_item(r)
        b.end_document()
    b.finalize(str(tmp_path / "d.idx"))
    ds = MMapIndexedDataset(str(tmp_path / "d"))
    assert len(ds) == 4 and all(np.array_equal(ds[i], rows[i]) for i in range(4))
    assert np.array_equal(ds.get(1, 2, 2), rows[1][2:4])

    class Lens(torch.utils.data.Dataset):
        lens = [3, 9, 5, 12, 7, 3, 10, 6]

        def __len__(self):
            return len(self.lens)

        def __getitem__(self, i):
            return torch.tensor(self.lens[i])

    an = DataAnalyzer(Lens(), num_workers=2, worker_id=0, batch_size=3, metric_names=["seqlen"],
                      metric_functions=[lambda batch: batch.numpy()], metric_types=["single_value_per_sample"],
                      metric_dtypes=[np.int64], save_path=str(tmp_path / "an"))
    an.run_map()
    an2 = DataAnalyzer(Lens(), num_workers=2, worker_id=1, batch_size=3, metric_names=["seqlen"],
                       metric_functions=[lambda batch: batch.numpy()], metric_types=["single_value_per_sample"],
                       metric_dtypes=[np.int64], save_path=str(tmp_path / "an"))
    an2.run_map()
    an.run_reduce()
    base = str(tmp_path / "an" / "seqlen" / "seqlen")
    i2m = MMapIndexedDataset(base + "_index_to_metric")
    assert [int(i2m[i][0]) for i in range(len(i2m))] == sorted(set(Lens.lens))
    cfg = {"seed": 1, "data_sampling": {"num_epochs": 2, "curriculum_learning": {"enabled": True, "curriculum_metrics": {
        "seqlen": {"index_to_sample_path": base + "_index_to_sample", "index_to_metric_path": base + "_index_to_metric",
                   "difficulty_type": "value", "clustering_type": "single_cluster", "min_difficulty": 5,
                   "max_difficulty": 12, "schedule_type": "fixed_linear",
                   "schedule_config": {"total_curriculum_step": 4, "difficulty_step": 1}}}}}}
    sampler = DeepSpeedDataSampler(cfg, 8, micro_batch_size=2, data_parallel_rank=0, data_parallel_size=1,
                                   data_parallel_group=None, gradient_accumulation_steps=1, global_rank=0)
    it = iter(sampler)
    first = next(it)
    assert all(Lens.lens[i] <= 5 for i in first)  # step 1: difficulty floor(5 + 7/4) = 6 -> lens <= 6
    for _ in range(4):
        batch = next(it)
    assert len(batch) == 2
    sd = sampler.state_dict()
    sampler.load_state_dict(sd)
    # range queries + the cluster view over the same index
    lens = np.asarray(Lens.lens)
    got = sampler.get_sample_based_on_metric_value("seqlen", 5, 8)
    assert sorted(got.tolist()) == sorted(np.nonzero((lens > 5) & (lens <= 8))[0].tolist())
    assert sampler.get_sample_based_on_metric_value("seqlen", 1000, 2000) is None
    everything = sampler.get_sample_based_on_metric_percentile("seqlen", 0, 12)  # the top of the scale closes the range
    assert sorted(everything.tolist()) == list(range(len(lens))) and list(lens[everything]) == sorted(lens)
    sampler.current_difficulties = {"seqlen": 6}
    assert sampler.get_new_cluster({}) and not sampler.get_new_cluster({"seqlen": 6})
    sampler.current_difficulties = {"seqlen": 12}
    assert sampler.get_new_cluster({"seqlen": 6})
    assert sum(sampler.data_cluster_sizes) == len(lens) and sampler.sample_from_clusters().sum() == sampler.global_batch_size
    n0 = sampler.data_cluster_sizes[0]
    drawn = sampler.get_sample_from_cluster(0, n0 + 1)  # wraps around after a reshuffle
    assert len(drawn) == n0 + 1 and set(drawn) == set(sampler.data_clusters[0].tolist())


def test_random_ltd_wrapper_and_scheduler():
    from deepspeed_b200.runtime.data_pipeline.data_routing import RandomLTDScheduler, convert_to_random_ltd
    from deepspeed_b200.runtime.data_pipeline.data_routing.helper import save_without_random_ltd

    class Block(nn.Module):
        def __init__(self):
            super().__init__()
            self.lin = nn.Linear(8, 8)

        def forward(self, x, attention_mask=None):
            return x + self.lin(x)

    model = nn.Sequential(Block(), Block())
    convert_to_random_ltd(model, Block)
    cfg = {"total_layer_num": 2, "random_ltd_layer_num": 2, "global_batch_size": 4, "model_mask_name": None,
           "micro_batch_size": 2, "hidden_state_order": "batch_seq_dim", "model_type": "decoder",
           "random_ltd_schedule": {"min_value": 4, "max_value": 10, "schedule_type": "fixed_linear",
                                   "schedule_config": {"seq_per_step": 2, "require_steps": 1}}}
    sched = RandomLTDScheduler(cfg)
    for i, m in enumerate(model):
        m.init_config(cfg, sched, i)
    sched.update_seq(0)
    assert sched.get_current_seq() == 4
    x = torch.randn(2, 10, 8, requires_grad=True)
    y = model.train()(x)
    assert y.shape == x.shape
    changed = (y - x).abs().sum(-1) > 0
    assert changed.sum(1).max() <= 8 and changed.sum(1).min() >= 4  # each layer touched 4 tokens
    y.sum().backward()
    assert torch.isfinite(x.grad).all()
    sched.update_seq(3)
    assert sched.get_current_seq() == 10
    assert all(".random_ltd_layer" not in k for k in save_without_random_ltd(model))


def test_indexed_dataset_formats_and_interop(tmp_path):
    import numpy as np
    import torch
    from deepspeed_b200.runtime.data_pipeline.data_sampling import indexed_dataset as I
    samples = [np.arange(5), np.arange(3) + 10, np.arange(7) + 100]
    # --- legacy TNTIDX: lazy + cached readers
    pre = str(tmp_path / "legacy")
    b = I.make_builder(I.data_file_path(pre), impl="cached", dtype=np.int32)
    for s in samples:
        b.add_item(torch.from_numpy(s))
        b.end_document()
    b.finalize(I.index_file_path(pre))
    assert I.infer_dataset_impl(pre) == "cached" and I.dataset_exists(pre, "cached")
    lazy = I.make_dataset(pre, "lazy")
    assert len(lazy) == 3 and all(np.array_equal(lazy[i], s) for i, s in enumerate(samples))
    assert [a.tolist() for a in lazy[0:2]] == [s.tolist() for s in samples[:2]]
    cached = I.make_dataset(pre, "infer")
    assert isinstance(cached, I.IndexedCachedDataset) and cached.supports_prefetch
    cached.prefetch([2, 0])
    assert np.array_equal(cached[2], samples[2]) and np.array_equal(cached[0], samples[0])
    # --- Megatron MMIDIDX written here
    meg = str(tmp_path / "meg")
    b = I.make_builder(I.data_file_path(meg), impl="mmap", dtype=np.uint16, fmt="megatron")
    for s in samples:
        b.add_item(s)
        b.end_document()
    b.finalize(I.index_file_path(meg))
    ds = I.make_dataset(meg, "infer")
    assert ds.dtype == np.uint16 and all(np.array_equal(ds[i], s) for i, s in enumerate(samples))
    assert I.code(np.int64) == 5 and I.code(torch.int16) == 3 and I.create_doc_idx([3, 0, 2, 0]) == [0, 2, 4]
    p, tot = I.get_pointers_with_total([2, 3, 4], 4, np.int64)
    assert p.tolist() == [0, 8, 20] and tot == 36
    # --- both directions against upstream DeepSpeed's indexed_dataset.py, through files its builders wrote for the same
    # samples (tests/golden/indexed_dataset, regenerate: scripts/make_reference_golden.py)
    import os
    golden = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden", "indexed_dataset")
    for prefix, theirs in ((meg, "mmap_uint16"), (pre, "legacy_int32")):  # upstream reads ours: the bytes are its own
        for ext in (".bin", ".idx"):
            with open(prefix + ext, "rb") as a, open(os.path.join(golden, theirs + ext), "rb") as b:
                assert a.read() == b.read(), theirs + ext
    mine = I.MMapIndexedDataset(os.path.join(golden, "mmap_int32"))
    assert mine.dtype == np.int32 and all(np.array_equal(mine[i], s) for i, s in enumerate(samples))
    assert mine.doc_idx.tolist() == ds.doc_idx.tolist()
    rl = I.make_dataset(os.path.join(golden, "legacy_int32"), "lazy")
    assert all(np.array_equal(rl[i], s) for i, s in enumerate(samples))


def _dist_helpers():
    import torch
    import deepspeed_b200 as ds
    from deepspeed_b200 import comm as dist
    from deepspeed_b200.runtime.data_pipeline.data_sampling.data_analyzer import Dist
    ds.init_distributed()
    r, w = dist.get_rank(), dist.get_world_size()
    t = torch.arange(3 + 2 * r, dtype=torch.int64) + 10 * r
    lo, hi = Dist.min_max(t.clone(), None)
    if r == 0:
        assert (lo, hi) == (0, 14)
    parts = Dist.gather_v(t, 0, None, w, r)
    if r == 0:
        assert [p.tolist() for p in parts] == [[0, 1, 2], [10, 11, 12, 13, 14]]
    else:
        assert parts is None
    g = torch.Generator().manual_seed(r)
    rows = torch.stack([torch.randint(0, 1000, (50, ), generator=g), torch.arange(50) + 100 * r], 1)
    mine = Dist.sample_sort(rows, None, w, n_samples=10)
    assert torch.all(mine[1:, 0] >= mine[:-1, 0])
    edge = torch.tensor([int(mine[0, 0]) if len(mine) else 10**9, int(mine[-1, 0]) if len(mine) else -1, len(mine)])
    allv = [torch.zeros_like(edge) for _ in range(w)]
    dist.all_gather(allv, edge)
    assert sum(int(v[2]) for v in allv) == 100 and int(allv[0][1]) <= int(allv[1][0])


def test_data_analyzer_dist_helpers():
    from tests.common import run_distributed
    run_distributed(_dist_helpers, 2)
