"""Checkpoint round trips: same-shape resume, zero_to_fp32 consolidation, universal checkpoint reshaping."""
import copy
import os

import pytest
import torch

from tests.common import run_distributed
from tests.unit.simple_model import SimpleModel, base_config, make_batch


def _steps(eng, n, seed, dtype="fp32"):
    import deepspeed_b200 as ds
    r, w = ds.comm.get_rank(), ds.comm.get_world_size()
    g = torch.Generator().manual_seed(seed)
    for _ in range(n):
        x, y = make_batch(2, 4, g)          # fixed global batch of 8 regardless of world size
        per = 8 // w
        loss = eng(x[r * per:(r + 1) * per], y[r * per:(r + 1) * per])
        eng.backward(loss)
        eng.step()
    return loss


def _cfg(stage, w):
    c = base_config(stage, "fp32", 1, 0.0)
    c["train_micro_batch_size_per_gpu"] = 8 // w
    c.pop("train_batch_size", None)
    return c


def _save_worker(d, stage):
    import deepspeed_b200 as ds
    torch.manual_seed(0)
    eng, *_ = ds.initialize(model=SimpleModel(), config=_cfg(stage, ds.comm.get_world_size()))
    _steps(eng, 3, 1)
    eng.save_checkpoint(d, tag="t3", client_state={"hello": 7})
    from deepspeed_b200.utils import safe_get_full_fp32_param
    at_save = {n: safe_get_full_fp32_param(p).cpu() for n, p in eng.module.named_parameters()}
    if ds.comm.get_rank() == 0:
        torch.save(at_save, os.path.join(d, "expect_at_save.pt"))
    # continue 2 more steps and record the parameters the resumed run must reproduce
    _steps(eng, 2, 2)
    full = {n: safe_get_full_fp32_param(p).cpu() for n, p in eng.module.named_parameters()}
    if ds.comm.get_rank() == 0:
        torch.save(full, os.path.join(d, "expect.pt"))


def _resume_worker(d, stage):
    import deepspeed_b200 as ds
    from deepspeed_b200.utils import safe_get_full_fp32_param
    torch.manual_seed(123)  # different init: everything must come from the checkpoint
    eng, *_ = ds.initialize(model=SimpleModel(), config=_cfg(stage, ds.comm.get_world_size()))
    path, client = eng.load_checkpoint(d)
    assert path is not None and client["hello"] == 7 and eng.global_steps == 3
    _steps(eng, 2, 2)
    exp = torch.load(os.path.join(d, "expect.pt"))
    for n, p in eng.module.named_parameters():
        torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("stage", [1, 3])
def test_save_resume_same_shape(tmp_path, stage):
    d = str(tmp_path)
    run_distributed(_save_worker, 2, (d, stage))
    run_distributed(_resume_worker, 2, (d, stage))


def _elastic_resume_worker(d, stage):
    """Resume at a different data-parallel degree than the checkpoint was written with, in-engine (no offline conversion)."""
    import deepspeed_b200 as ds
    from deepspeed_b200.utils import safe_get_full_fp32_param, safe_get_full_optimizer_state
    torch.manual_seed(77)
    eng, *_ = ds.initialize(model=SimpleModel(), config=_cfg(stage, ds.comm.get_world_size()))
    path, client = eng.load_checkpoint(d)
    assert path is not None and client["hello"] == 7 and eng.global_steps == 3
    at_save = torch.load(os.path.join(d, "expect_at_save.pt"))
    for n, p in eng.module.named_parameters():
        torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), at_save[n], atol=0, rtol=0)
        m = safe_get_full_optimizer_state(p, "exp_avg")
        assert m is not None and m.abs().sum() > 0, "optimizer moments must be restored too"
    _steps(eng, 2, 2)
    exp = torch.load(os.path.join(d, "expect.pt"))
    for n, p in eng.module.named_parameters():
        torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=2e-6, rtol=1e-5)


@pytest.mark.parametrize("stage,saved_world,new_world", [(1, 2, 1), (2, 2, 4), (3, 2, 1), (3, 1, 2)])
def test_resume_at_a_different_dp_degree(tmp_path, stage, saved_world, new_world):
    d = str(tmp_path)
    run_distributed(_save_worker, saved_world, (d, stage))
    run_distributed(_elastic_resume_worker, new_world, (d, stage))


def _universal_resume_worker(d, stage):
    import deepspeed_b200 as ds
    from deepspeed_b200.utils import safe_get_full_fp32_param
    torch.manual_seed(321)
    c = _cfg(stage, ds.comm.get_world_size())
    c["checkpoint"] = {"load_universal": True}
    eng, *_ = ds.initialize(model=SimpleModel(), config=c)
    eng.load_checkpoint(d, tag="t3_universal")
    assert eng.global_steps == 3
    _steps(eng, 2, 2)
    exp = torch.load(os.path.join(d, "expect.pt"))
    for n, p in eng.module.named_parameters():
        torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=1e-5, rtol=1e-4)


def test_zero_to_fp32_and_universal_reshape(tmp_path):
    d = str(tmp_path)
    run_distributed(_save_worker, 2, (d, 3))
    # (a) offline consolidation script (copied next to the checkpoint) reproduces the saved weights
    assert os.path.isfile(os.path.join(d, "zero_to_fp32.py"))
    from deepspeed_b200.utils.zero_to_fp32 import get_fp32_state_dict_from_zero_checkpoint, \
        convert_zero_checkpoint_to_fp32_state_dict
    sd = get_fp32_state_dict_from_zero_checkpoint(d)
    m = SimpleModel()
    m.load_state_dict(sd, strict=True)
    convert_zero_checkpoint_to_fp32_state_dict(d, os.path.join(d, "out"), max_shard_size="1KB")
    assert any(f.endswith(".index.json") for f in os.listdir(os.path.join(d, "out")))
    # (b) universal: saved with dp=2 stage 3, resumed with dp=1 stage 2 and dp=3 stage 1; both reproduce the run
    from deepspeed_b200.checkpoint import convert_to_universal
    convert_to_universal(os.path.join(d, "t3"), os.path.join(d, "t3_universal"))
    run_distributed(_universal_resume_worker, 1, (d, 2))


def test_reshape_2d_and_3d_maps():
    from deepspeed_b200.checkpoint import get_mpu_ranks, model_3d_desc, reshape_meg_2d_parallel
    g = reshape_meg_2d_parallel(old_pp_degree=2, old_tp_degree=4, new_pp_degree=1, new_tp_degree=2)
    # source rank = pp*4 + tp; tp 4->2 merges (0,1),(2,3); pp 2->1 stacks the stages
    assert g.get_data(0, 0) == [0, 1, 4, 5] and g.get_data(0, 1) == [2, 3, 6, 7]
    maps = model_3d_desc(pp_degree=1, tp_degree=2, dp_degree=4).reshape(model_3d_desc(1, 1, 2))
    assert len(maps) == 2
    assert sorted(maps[0].get_data(0, 0) + maps[1].get_data(0, 0)) == list(range(8))
    ok, errs = model_3d_desc(1, 1, 2).can_reshape(model_3d_desc(1, 2, 2))
    assert not ok and "TP" in errs[0]
    tp, pp, dp = get_mpu_ranks(tp_size=2, pp_size=4, dp_size=2)
    assert tp[0] == [0, 1] and dp[0] == [0, 2] and pp[0] == [0, 4, 8, 12] and pp[1] == [1, 5, 9, 13]


def test_zero_checkpoint_merge(tmp_path):
    import torch
    from deepspeed_b200.checkpoint import ZeROCheckpoint, model_3d_desc
    from deepspeed_b200.checkpoint.constants import (BASE_OPTIMIZER_STATE, GROUP_PADDINGS, OPTIMIZER_STATE_DICT,
                                                     PARTITION_COUNT)
    d = tmp_path / "global_step1"
    d.mkdir()
    torch.save({}, d / "mp_rank_00_model_states.pt")
    for dp in range(4):
        pad = 2 if dp == 3 else 0
        flat = torch.arange(dp * 6, dp * 6 + 6, dtype=torch.float32)
        sd = {OPTIMIZER_STATE_DICT: {BASE_OPTIMIZER_STATE: {"state": {0: {"exp_avg": flat.clone(), "step": 5}}},
                                     GROUP_PADDINGS: [pad], PARTITION_COUNT: [4]}}
        torch.save(sd, d / f"zero_pp_rank_{dp}_mp_rank_00_optim_states.pt")
    z = ZeROCheckpoint(str(d))
    assert (z.get_src_dp_degree(), z.get_src_tp_degree(), z.get_src_pp_degree()) == (4, 1, 1)
    z.reshape(model_3d_desc(1, 1, 2))
    a = z.get_state_for_rank(0, 0, 0)[OPTIMIZER_STATE_DICT]
    b = z.get_state_for_rank(0, 0, 1)[OPTIMIZER_STATE_DICT]
    assert a[BASE_OPTIMIZER_STATE]["state"][0]["exp_avg"].tolist() == list(map(float, range(12)))
    assert b[BASE_OPTIMIZER_STATE]["state"][0]["exp_avg"].tolist() == list(map(float, range(12, 22)))  # padding stripped
    assert a[PARTITION_COUNT] == [2] and b[GROUP_PADDINGS] == [0]


def test_nebula_tiered_engine(tmp_path):
    import os
    import torch
    from deepspeed_b200.nebula.config import DeepSpeedNebulaConfig
    from deepspeed_b200.runtime.checkpoint_engine import NebulaCheckpointEngine
    fast, slow = tmp_path / "fast", tmp_path / "slow"
    cfg = DeepSpeedNebulaConfig({"nebula": {"enabled": True, "persistent_storage_path": str(slow),
                                            "persistent_time_interval": 0, "num_of_version_in_retention": 2}})
    eng = NebulaCheckpointEngine(cfg)
    for step in range(4):
        tag = f"global_step{step}"
        os.makedirs(fast / tag)
        eng.create(tag)
        eng.save({"w": torch.full((3, ), float(step))}, str(fast / tag / "mp_rank_00_model_states.pt"))
        eng.commit(tag)
        eng.wait_persisted()
    kept = sorted(d for d in os.listdir(slow) if os.path.isdir(slow / d))
    assert kept == ["global_step2", "global_step3"] and (slow / "latest").read_text() == "global_step3"
    # the fast tier lost a version: load falls back to the persistent copy
    os.remove(fast / "global_step3" / "mp_rank_00_model_states.pt")
    sd = eng.load(str(fast / "global_step3" / "mp_rank_00_model_states.pt"))
    assert sd["w"].tolist() == [3.0, 3.0, 3.0]


def _write_upstream_ckpt(root, stage, world, with_frozen=True):
    """Hand-build a checkpoint in the upstream DeepSpeed on-disk layout (what ``zero_to_fp32`` of the reference reads)."""
    import math
    import os
    import torch
    torch.manual_seed(stage)
    groups = [{"a.weight": torch.Size([5, 3]), "a.bias": torch.Size([5])}, {"b.weight": torch.Size([7, 2])}]
    full = {k: torch.randn(*shp) for g in groups for k, shp in g.items()}
    frozen = {"f.weight": torch.randn(4, 3)} if with_frozen else {}
    buf = {"bn.running_mean": torch.arange(4.0)}
    tag = "global_step5"
    d = os.path.join(root, tag)
    os.makedirs(d)
    with open(os.path.join(root, "latest"), "w") as f:
        f.write(tag)
    if stage <= 2:
        align = 2 * world
        per_rank = [[] for _ in range(world)]
        for g in groups:
            flat = torch.cat([full[k].reshape(-1) for k in g])
            padded = align * math.ceil(flat.numel() / align)
            flat = torch.cat([flat, torch.zeros(padded - flat.numel())])
            for r, piece in enumerate(flat.chunk(world)):
                per_rank[r].append(piece.clone())
        key = "single_partition_of_fp32_groups"
        model_files = ["mp_rank_00_model_states.pt"]
    else:
        # stage 3: every parameter is split over the ranks; a rank's groups are back-to-back slices (a parameter may even
        # straddle two sub-groups: put the boundary in the middle of a.bias)
        names = [k for g in groups for k in g]
        per_rank_flat = []
        for r in range(world):
            pieces = []
            for k in names:
                n = full[k].numel()
                per = math.ceil(n / world)
                padded = torch.cat([full[k].reshape(-1), torch.zeros(per * world - n)])
                pieces.append(padded[r * per:(r + 1) * per])
            per_rank_flat.append(torch.cat(pieces))
        cut = math.ceil(15 / world) + 1
        per_rank = [[f[:cut].clone(), f[cut:].clone()] for f in per_rank_flat]
        key = "fp32_flat_groups"
        model_files = [f"zero_pp_rank_{r}_mp_rank_00_model_states.pt" for r in range(world)]
    for r in range(world):
        torch.save({"optimizer_state_dict": {"zero_stage": stage, "partition_count": world, key: per_rank[r],
                                             "optimizer_state_dict": {"state": {}}}},
                   os.path.join(d, f"zero_pp_rank_{r}_mp_rank_00_optim_states.pt"))
    for r, mf in enumerate(model_files):
        if stage <= 2:
            frags = dict(frozen)
        else:
            frags = {}
            for k, v in frozen.items():
                per = math.ceil(v.numel() / world)
                padded = torch.cat([v.reshape(-1), torch.zeros(per * world - v.numel())])
                frags[k] = padded[r * per:(r + 1) * per].clone()
        torch.save({"module": dict(buf), "buffer_names": list(buf), "param_shapes": groups,
                    "shared_params": {"tied.weight": "a.weight"}, "ds_version": "0.16.5",
                    "frozen_param_shapes": {k: v.shape for k, v in frozen.items()} or None,
                    "frozen_param_fragments": frags or None}, os.path.join(d, mf))
    expect = dict(full, **frozen, **buf)
    expect["tied.weight"] = full["a.weight"]
    return expect


@pytest.mark.parametrize("stage,world", [(2, 2), (1, 3), (3, 2), (3, 4)])
def test_zero_to_fp32_reads_upstream_layout(tmp_path, stage, world):
    import torch
    from deepspeed_b200.utils import zero_to_fp32 as Z
    expect = _write_upstream_ckpt(str(tmp_path), stage, world)
    sd = Z.get_fp32_state_dict_from_zero_checkpoint(str(tmp_path))
    assert set(sd) == set(expect)
    for k, v in expect.items():
        assert torch.equal(sd[k].float(), v.float()), k
    no_frozen = Z.get_fp32_state_dict_from_zero_checkpoint(str(tmp_path), exclude_frozen_parameters=True)
    assert "f.weight" not in no_frozen
    lazy = Z.get_fp32_state_dict_from_zero_checkpoint(str(tmp_path), lazy_mode=True)
    if stage == 3:
        assert isinstance(lazy["a.bias"], Z.GatheredTensor) and torch.equal(lazy["a.bias"].contiguous(), expect["a.bias"])
        assert Z.zero3_partitioned_param_info(15, 4) == (4, 1)
    out = tmp_path / "out"
    Z.convert_zero_checkpoint_to_fp32_state_dict(str(tmp_path), str(out))
    got = torch.load(out / "pytorch_model.bin")
    assert torch.equal(got["b.weight"], expect["b.weight"])
    assert Z.natural_keys("rank_10") > Z.natural_keys("rank_9")
    assert Z.get_model_state_file(str(tmp_path / "global_step5"), stage).endswith("model_states.pt")


def test_ds_to_universal_staged_pipeline(tmp_path):
    """Upstream stage-3 checkpoint → fragments → universal; and TP-slice merge rules round-trip through the loader."""
    import math
    import os
    import torch
    from deepspeed_b200.checkpoint import ds_to_universal as U
    from deepspeed_b200.checkpoint import constants as K
    from deepspeed_b200.checkpoint.universal_checkpoint import load_hp_checkpoint_state, SubparamShape, enable_universal_checkpoint
    # ---- stage 3, upstream layout, dp=3
    dp = 3
    shapes = {"w": torch.Size([4, 5]), "b": torch.Size([7])}
    full = {s: {k: torch.randn(*shp) for k, shp in shapes.items()} for s in ("fp32", "exp_avg", "exp_avg_sq")}
    src = tmp_path / "global_step1"
    os.makedirs(src)
    for r in range(dp):
        flat = {}
        for s in full:
            parts = []
            for k, shp in shapes.items():
                n = shp.numel()
                per = math.ceil(n / dp)
                padded = torch.cat([full[s][k].reshape(-1), torch.zeros(per * dp - n)])
                parts.append(padded[r * per:(r + 1) * per])
            flat[s] = torch.cat(parts)
        torch.save({"optimizer_state_dict": {"zero_stage": 3, "partition_count": dp, "fp32_flat_groups": [flat["fp32"]],
                                             "optimizer_state_dict": {"state": {0: {"exp_avg": flat["exp_avg"],
                                                                                  "exp_avg_sq": flat["exp_avg_sq"]}}}}},
                   src / f"zero_pp_rank_{r}_mp_rank_00_optim_states.pt")
        torch.save({"module": {}, "buffer_names": [], "param_shapes": [shapes], "shared_params": {}, "ds_version": "0.16.5"},
                   src / f"zero_pp_rank_{r}_mp_rank_00_model_states.pt")
    out = tmp_path / "universal"
    U.main(U.parse_arguments(["--input_folder", str(src), "--output_folder", str(out)]))
    for s in full:
        for k, shp in shapes.items():
            got = load_hp_checkpoint_state(str(out / "zero" / k), s, shp)
            assert torch.equal(got, full[s][k]), (s, k)
    assert not (out / "tmp").exists() and U.dp_index_to_str(3) == "03"
    # ---- TP merge rules: write per-(tp, dp) fragments by hand, merge, then re-slice with the loader
    tp, tmp2, dst = 2, str(tmp_path / "frags"), str(tmp_path / "merged")
    info = {K.UNIVERSAL_CHECKPOINT_INFO: {}}
    rules = {K.TP_REPLICATED_PARAMETER_PATTERNS: [r"ln\."], K.PARAMETER_WITH_ROW_PARALLELISM_PATTERNS: [r"row\."],
             K.PARAMETER_WITH_2_SUB_PARAMS_CAT_DIM_0: [r"glu\."], K.VOCABULARY_PARAMETER_PATTERNS: [r"emb\."],
             K.ORIGINAL_VOCAB_SIZE: 5,
             K.PARAMETER_WITH_SUB_PARAMS: [dict(patterns=[r"qkv\."], shape=((4, 2, 2), 3), partition_dim=0)]}

    class _Ck:

        def get_checkpoint_info(self, key=None):
            return rules

    fulls = {"ln.w": torch.randn(6), "row.w": torch.randn(3, 8), "col.w": torch.randn(8, 3), "glu.w": torch.randn(8, 3),
             "emb.w": torch.cat([torch.randn(5, 4), torch.zeros(1, 4)]), "qkv.w": torch.randn(8, 3)}

    def tp_slices(name, t):
        if name.startswith("ln"):
            return [t, t]
        if name.startswith("row"):
            return list(t.chunk(2, dim=1))
        if name.startswith("glu"):
            a, b = t.chunk(2, 0)
            return [torch.cat([a.chunk(2, 0)[r], b.chunk(2, 0)[r]]) for r in range(2)]
        if name.startswith("qkv"):
            q, k, v = t.split([4, 2, 2], 0)
            return [torch.cat([x.chunk(2, 0)[r] for x in (q, k, v)]) for r in range(2)]
        return list(t.chunk(2, dim=0))

    for name, t in fulls.items():
        for r, sl in enumerate(tp_slices(name, t)):
            flat = sl.reshape(-1)
            half = flat.numel() // 2
            for st in ("fp32", "exp_avg", "exp_avg_sq"):
                U.dump_param_fragment(tmp2, r, 0, st, flat, name, 0, half)
                U.dump_param_fragment(tmp2, r, 1, st, flat, name, half, flat.numel() - half)
            U.dump_param_fragment(tmp2, r, 0, "step", torch.tensor(7.0), name, 0, 0)
    unmatched = set()
    for name, t in fulls.items():
        sl_shape = tp_slices(name, t)[0].shape
        unmatched |= U.merge_tp_slices(_Ck(), dst, tmp2, tp, (name, sl_shape)) if name == "ln.w" else set()
        if name != "ln.w":
            U.merge_tp_slices(_Ck(), dst, tmp2, tp, (name, sl_shape))
    for name, t in fulls.items():
        merged = torch.load(os.path.join(dst, name, "fp32.pt"), weights_only=False)
        want = t[:5] if name == "emb.w" else t
        assert torch.equal(merged["param"], want), name
        # loading back at tp=2 recovers each rank's slice
        for r, sl in enumerate(tp_slices(name, t)):
            got = load_hp_checkpoint_state(os.path.join(dst, name), "fp32", sl.shape, tp_rank=r, tp_world_size=2)
            assert torch.equal(got, sl), (name, r)
    assert float(torch.load(os.path.join(dst, "ln.w", "step.pt"), weights_only=False)) == 7.0
    p = torch.nn.Parameter(torch.zeros(8, 3))
    enable_universal_checkpoint([p])
    assert torch.equal(p.load_hp_checkpoint_state(os.path.join(dst, "col.w")), fulls["col.w"])
    assert SubparamShape(patterns=["x"], shape=(1, ), partition_dim=0).partition_dim == 0


def test_deepspeed_checkpoint_layer_file_maps(tmp_path):
    import torch
    from deepspeed_b200.checkpoint import DeepSpeedCheckpoint
    d = tmp_path / "global_step3"
    d.mkdir()
    for layer in (1, 3, 4, 5, 6, 8):  # embedding, 4 transformer layers, final norm
        for tp in range(2):
            torch.save({"w": torch.full((2, 3), float(10 * layer + tp))}, d / f"layer_{layer:02d}-model_{tp:02d}-model_states.pt")
    for pp in range(2):
        for tp in range(2):
            torch.save({"global_steps": 3, "args": {"a": 1}, "module": {"x": torch.full((1, ), float(pp * 2 + tp))}},
                       d / f"mp_rank_{pp * 2 + tp:02d}_model_states.pt")
    ck = DeepSpeedCheckpoint(str(d), tp_degree=2, pp_degree=2)
    assert ck.original_tp_degree in (2, 4)  # without zero files the tp/pp split of mp_rank files is ambiguous
    ck.original_tp_degree, ck.original_pp_degree, ck._maps = 2, 2, None
    assert ck.get_embedding_layer_id() == "layer_01" and ck.get_final_norm_layer_id() == "layer_08"
    assert ck.get_pp_transformer_map(0) == ["layer_03", "layer_04"] and ck.get_pp_transformer_map(1) == ["layer_05", "layer_06"]
    assert [f.split("/")[-1] for f in ck.get_embedding_files(1)] == ["layer_01-model_01-model_states.pt"]
    st = ck.get_transformer_state(tp_index=1, pp_index=1)
    assert len(st) == 2 and float(st[0]["w"][0, 0]) == 51.0 and float(st[1]["w"][0, 0]) == 61.0
    assert float(ck.get_final_norm_state(0)["w"][0, 0]) == 80.0 and float(ck.get_embedding_state(0)["w"][0, 0]) == 10.0
    assert len(ck.get_2d_parallel_files(tp_index=1, pp_index=0)) == 1 and ck.get_iteration() == 3 and ck.validate_files()
    # contraction tp 2 -> 1: the two TP slices of a layer are merged
    ck1 = DeepSpeedCheckpoint(str(d), tp_degree=1, pp_degree=2)
    ck1.original_tp_degree, ck1.original_pp_degree, ck1._maps = 2, 2, None
    merged = ck1.get_transformer_state(tp_index=0, pp_index=0)[0]["w"]
    assert merged.shape == (4, 3) and merged[:, 0].tolist() == [30.0, 30.0, 31.0, 31.0]
    assert len(ck1.get_2d_parallel_files(tp_index=0, pp_index=1)) == 2
    ck1.show_pp_transformer_map()


# ---- interop with UNMODIFIED upstream DeepSpeed, both directions -----------------------------------------------------
# What upstream saved or consolidated is stored under tests/golden/ (regenerate: scripts/make_reference_golden.py).
_GOLDEN = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden")

# the script upstream ran (gloo ws=2) to write tests/golden/ref_ckpt_stage{2,3}
_REF_SAVE = r'''
import os, sys
sys.path.insert(0, {ref!r})
os.environ.setdefault("DS_ACCELERATOR", "cpu")
import torch, torch.distributed as dist
import deepspeed
sys.path.insert(0, {root!r})
from tests.unit.simple_model import SimpleModel, make_batch
out, stage = sys.argv[1], int(sys.argv[2])
deepspeed.init_distributed(dist_backend="gloo")
r, w = dist.get_rank(), dist.get_world_size()
torch.manual_seed(0)
model = SimpleModel()
cfg = {{"train_micro_batch_size_per_gpu": 4, "zero_optimization": {{"stage": stage, "stage3_param_persistence_threshold": 0}},
       "zero_allow_untested_optimizer": True, "zero_force_ds_cpu_optimizer": False}}
opt = torch.optim.AdamW(model.parameters(), lr=1e-2, weight_decay=0.01)
eng, *_ = deepspeed.initialize(model=model, optimizer=opt, config=cfg)
g = torch.Generator().manual_seed(1)
def steps(n):
    for _ in range(n):
        x, y = make_batch(w, 4, g)
        eng.backward(eng(x[r*4:(r+1)*4], y[r*4:(r+1)*4])); eng.step()
steps(3)
eng.save_checkpoint(out, tag="ref3", client_state={{"hello": 7}})
steps(2)
from deepspeed.utils import safe_get_full_fp32_param
full = {{n: safe_get_full_fp32_param(p).detach().cpu().clone() for n, p in eng.module.named_parameters()}}
if r == 0:
    torch.save(full, os.path.join(out, "expect_after5.pt"))
dist.barrier()
'''


def _assert_same_checkpoint_object(got, want, where):
    """``got`` holds what ``want`` holds, in the same order (dict keys, lists, ``param_shapes``): tensors equal in dtype,
    shape and value (within the tolerance of the resume tests), every other leaf equal.  ``ds_version`` is not compared."""
    assert type(got) is type(want), f"{where}: {type(got).__name__} != {type(want).__name__}"
    if isinstance(want, dict):
        assert list(got) == list(want), f"{where}: keys {list(got)} != {list(want)}"
        for k in want:
            if k != "ds_version":
                _assert_same_checkpoint_object(got[k], want[k], f"{where}/{k}")
    elif isinstance(want, (list, tuple)):
        assert len(got) == len(want), f"{where}: length {len(got)} != {len(want)}"
        for i, (g, w) in enumerate(zip(got, want)):
            _assert_same_checkpoint_object(g, w, f"{where}[{i}]")
    elif torch.is_tensor(want):
        assert got.dtype == want.dtype and got.shape == want.shape, f"{where}: {got.dtype}{list(got.shape)} != " \
            f"{want.dtype}{list(want.shape)}"
        torch.testing.assert_close(got, want, atol=1e-6, rtol=1e-5, msg=lambda m: f"{where}: {m}")
    elif isinstance(want, float):
        assert got == pytest.approx(want, rel=1e-5, abs=1e-6), f"{where}: {got} != {want}"
    elif hasattr(want, "__dict__"):
        _assert_same_checkpoint_object(vars(got), vars(want), where)
    else:
        assert got == want, f"{where}: {got!r} != {want!r}"


def _resume_from_ref_worker(d, stage):
    import deepspeed_b200 as ds
    from deepspeed_b200.utils import safe_get_full_fp32_param
    torch.manual_seed(123)  # different init: everything must come from the stock checkpoint
    cfg = {"train_micro_batch_size_per_gpu": 4, "optimizer": {"type": "AdamW", "params": {"lr": 1e-2, "weight_decay": 0.01}},
           "zero_optimization": {"stage": stage, "stage3_param_persistence_threshold": 0}}
    eng, *_ = ds.initialize(model=SimpleModel(), config=cfg)
    path, client = eng.load_checkpoint(d, tag="ref3")
    assert path is not None and client["hello"] == 7 and eng.global_steps == 3
    r, w = ds.comm.get_rank(), ds.comm.get_world_size()
    g = torch.Generator().manual_seed(1)
    for _ in range(3):
        make_batch(w, 4, g)  # the batches the reference run consumed before saving
    for _ in range(2):
        x, y = make_batch(w, 4, g)
        eng.backward(eng(x[r * 4:(r + 1) * 4], y[r * 4:(r + 1) * 4]))
        eng.step()
    exp = torch.load(os.path.join(d, "expect_after5.pt"))
    for n, p in eng.module.named_parameters():
        torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=2e-6, rtol=1e-5)


@pytest.mark.parametrize("stage", [2, 3])
def test_resume_in_engine_from_stock_deepspeed_checkpoint(stage):
    """(i) unmodified upstream DeepSpeed trained 3 steps on gloo ws=2 and saved; this engine resumes from those files and
    its next 2 steps land on upstream's own continuation."""
    run_distributed(_resume_from_ref_worker, 2, (os.path.join(_GOLDEN, f"ref_ckpt_stage{stage}"), stage))


@pytest.mark.parametrize("stage", [1, 3])
def test_stock_zero_to_fp32_reads_our_checkpoint(tmp_path, stage):
    """(ii) upstream's own ``zero_to_fp32.py`` consolidated the stored checkpoint files (saved here) into the stored
    weights: a checkpoint saved now holds what those files hold, and those weights are the engine's."""
    d = str(tmp_path)
    run_distributed(_save_worker, 2, (d, stage))
    golden = os.path.join(_GOLDEN, f"zero_to_fp32_stage{stage}")
    files = sorted(f for f in os.listdir(os.path.join(golden, "t3")) if f.endswith(".pt"))
    assert files and files == sorted(f for f in os.listdir(os.path.join(d, "t3")) if f.endswith(".pt"))
    for f in files:
        _assert_same_checkpoint_object(torch.load(os.path.join(d, "t3", f), map_location="cpu", weights_only=False),
                                       torch.load(os.path.join(golden, "t3", f), map_location="cpu", weights_only=False),
                                       f)
    got = torch.load(os.path.join(golden, "consolidated.pt"))
    exp = torch.load(os.path.join(d, "expect_at_save.pt"))
    assert set(exp) <= set(got)
    for n, v in exp.items():
        torch.testing.assert_close(got[n].float(), v, atol=1e-6, rtol=1e-5)


def _moe_ckpt_worker(d, phase):
    """Expert-parallel MoE checkpoint: dense weights in the model-states file, every expert in its own
    ``layer_#_expert_#_mp_rank_##_model_states.pt`` (reference ``engine.py:3376 _save_moe_checkpoint``), the dense and the
    expert optimizer domains in the ZeRO shard files.  A fresh engine resumed from it continues identically."""
    import deepspeed_b200 as ds
    from deepspeed_b200.models.mixtral import MixtralForCausalLM, mixtral_config
    from deepspeed_b200.utils import safe_get_full_fp32_param
    w, r = ds.comm.get_world_size(), ds.comm.get_rank()
    torch.manual_seed(0 if phase == "save" else 99)
    cfg = mixtral_config("tiny-moe", ep_size=w)
    eng, *_ = ds.initialize(model=MixtralForCausalLM(cfg), config={
        "train_micro_batch_size_per_gpu": 2, "optimizer": {"type": "AdamW", "params": {"lr": 2e-3}},
        "zero_optimization": {"stage": 1}})
    g = torch.Generator().manual_seed(11)
    batches = [torch.randint(0, cfg.vocab_size, (2 * w, 32), generator=g)[r * 2:(r + 1) * 2] for _ in range(5)]

    def run(lo, hi):
        for ids in batches[lo:hi]:
            eng.backward(eng(ids, labels=ids))
            eng.step()

    if phase == "save":
        run(0, 3)
        eng.save_checkpoint(d, tag="moe")
        ds.comm.barrier()
        files = os.listdir(os.path.join(d, "moe"))
        assert any(f.startswith("layer_") and "_expert_" in f for f in files), files
        run(3, 5)
        torch.save({n: safe_get_full_fp32_param(p).cpu() for n, p in eng.module.named_parameters()},
                   os.path.join(d, f"expect_rank{r}.pt"))
    else:
        path, _ = eng.load_checkpoint(d, tag="moe")
        assert path is not None and eng.global_steps == 3
        run(3, 5)
        exp = torch.load(os.path.join(d, f"expect_rank{r}.pt"))
        for n, p in eng.module.named_parameters():  # experts are rank-local: compared per rank
            torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=2e-6, rtol=1e-5, msg=n)


def test_moe_expert_parallel_checkpoint_resume(tmp_path):
    d = str(tmp_path)
    run_distributed(_moe_ckpt_worker, 2, (d, "save"))
    run_distributed(_moe_ckpt_worker, 2, (d, "load"))


def _pipe_ckpt_worker(d, phase):
    """Pipeline checkpoint: one ``layer_XX-model_states.pt`` per layer (reference ``pipe/module.py:605 save_state_dict``),
    loadable by a fresh 2-stage engine; training continues identically."""
    import deepspeed_b200 as ds
    from torch import nn
    from deepspeed_b200.pipe import PipelineModule
    from deepspeed_b200.utils import safe_get_full_fp32_param

    class Blk(nn.Module):

        def __init__(self, dd):
            super().__init__()
            self.l = nn.Linear(dd, dd)

        def forward(self, x):
            return torch.tanh(self.l(x))

    torch.manual_seed(0 if phase == "save" else 5)
    dd, micro, mbs = 16, 2, 2
    model = PipelineModule(layers=[Blk(dd) for _ in range(4)], num_stages=2, loss_fn=nn.MSELoss(), partition_method="uniform")
    eng, *_ = ds.initialize(model=model, config={"train_micro_batch_size_per_gpu": mbs, "gradient_accumulation_steps": micro,
                                                 "optimizer": {"type": "Adam", "params": {"lr": 1e-2}},
                                                 "zero_optimization": {"stage": 0}})
    g = torch.Generator().manual_seed(5)
    data = [[(torch.randn(mbs, dd, generator=g), torch.randn(mbs, dd, generator=g)) for _ in range(micro)] for _ in range(4)]
    own = {n: p for n, p in model.named_parameters()}
    if phase == "save":
        for it in range(2):
            eng.train_batch(data_iter=iter(data[it]))
        eng.save_checkpoint(d, tag="pp")
        ds.comm.barrier()
        files = os.listdir(os.path.join(d, "pp"))
        assert sum(f.startswith("layer_") and f.endswith("model_states.pt") for f in files) == 4, files
        for it in range(2, 4):
            eng.train_batch(data_iter=iter(data[it]))
        torch.save({n: safe_get_full_fp32_param(p).cpu() for n, p in own.items()},
                   os.path.join(d, f"expect_stage{eng.stage_id}.pt"))
    else:
        path, _ = eng.load_checkpoint(d, tag="pp")
        assert path is not None and eng.global_steps == 2
        for it in range(2, 4):
            eng.train_batch(data_iter=iter(data[it]))
        exp = torch.load(os.path.join(d, f"expect_stage{eng.stage_id}.pt"))
        for n, p in own.items():
            torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=2e-6, rtol=1e-5, msg=n)


def test_pipeline_layer_checkpoint_resume(tmp_path):
    d = str(tmp_path)
    run_distributed(_pipe_ckpt_worker, 2, (d, "save"))
    run_distributed(_pipe_ckpt_worker, 2, (d, "load"))


def _sched_ckpt_worker(d):
    """LR scheduler state, ``latest`` tag file and client state ride the checkpoint (reference ``engine.py:3218-3290``)."""
    import deepspeed_b200 as ds
    cfg = base_config(1, "fp32", 1, 0.0)
    cfg["scheduler"] = {"type": "WarmupLR", "params": {"warmup_min_lr": 0.0, "warmup_max_lr": 1e-2, "warmup_num_steps": 10}}
    torch.manual_seed(0)
    eng, _, _, sched = ds.initialize(model=SimpleModel(), config=cfg)
    _steps(eng, 4, 1)
    lr_at_save = eng.get_lr()[0]
    eng.save_checkpoint(d, client_state={"epoch": 3})  # default tag global_step4 + 'latest'
    assert open(os.path.join(d, "latest")).read().strip() == "global_step4"
    _steps(eng, 2, 2)
    assert eng.get_lr()[0] > lr_at_save
    torch.manual_seed(9)
    eng2, _, _, sched2 = ds.initialize(model=SimpleModel(), config=cfg)
    path, client = eng2.load_checkpoint(d)  # resolves 'latest'
    assert path is not None and "global_step4" in path and client["epoch"] == 3
    assert eng2.global_steps == 4 and abs(eng2.get_lr()[0] - lr_at_save) < 1e-12
    _steps(eng2, 2, 2)
    assert abs(eng2.get_lr()[0] - eng.get_lr()[0]) < 1e-12
    path3, _ = eng2.load_checkpoint(d, tag="does_not_exist")
    assert path3 is None


def test_scheduler_state_latest_tag_and_client_state(tmp_path):
    run_distributed(_sched_ckpt_worker, 1, (str(tmp_path), ))


def _frozen_model(seed):
    torch.manual_seed(seed)
    m = SimpleModel()
    first = next(iter(m.parameters()))
    first.requires_grad_(False)
    return m


def _frozen_ckpt_worker(d, stage, phase):
    import deepspeed_b200 as ds
    from deepspeed_b200.utils import safe_get_full_fp32_param
    from deepspeed_b200.utils.zero_to_fp32 import get_fp32_state_dict_from_zero_checkpoint
    if phase == "save":
        eng, *_ = ds.initialize(model=_frozen_model(0), config=_cfg(stage, ds.comm.get_world_size()))
        _steps(eng, 2, 1)
        eng.save_checkpoint(d, tag="fz")
        full = {n: safe_get_full_fp32_param(p).cpu() for n, p in eng.module.named_parameters()}
        ds.comm.barrier()
        if ds.comm.get_rank() == 0:
            torch.save(full, os.path.join(d, "expect.pt"))
            sd = get_fp32_state_dict_from_zero_checkpoint(d, "fz")
            for n, v in full.items():
                torch.testing.assert_close(sd[n].float(), v, atol=1e-6, rtol=1e-5)
        return
    eng, *_ = ds.initialize(model=_frozen_model(77), config=_cfg(stage, ds.comm.get_world_size()))
    path, _ = eng.load_checkpoint(d)
    assert path is not None
    exp = torch.load(os.path.join(d, "expect.pt"))
    for n, p in eng.module.named_parameters():
        torch.testing.assert_close(safe_get_full_fp32_param(p).cpu(), exp[n], atol=1e-6, rtol=1e-5)


@pytest.mark.parametrize("stage,new_world", [(2, 2), (3, 2), (3, 1)])
def test_frozen_parameters_round_trip(tmp_path, stage, new_world):
    """Frozen parameters live outside the optimizer shards: saved as reference-layout fragments next to the module state,
    restored in-engine (also at another DP degree) and read back by zero_to_fp32."""
    d = str(tmp_path)
    run_distributed(_frozen_ckpt_worker, 2, (d, stage, "save"))
    run_distributed(_frozen_ckpt_worker, new_world, (d, stage, "load"))
