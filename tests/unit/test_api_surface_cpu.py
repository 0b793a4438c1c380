"""Reference API names that user code imports directly: presence + behaviour of the small helpers."""
import argparse

import pytest
import torch

from tests.common import run_distributed


def test_top_level_and_lr_cli_helpers():
    import deepspeed_b200 as ds
    from deepspeed_b200.runtime import lr_schedules as L
    assert ds.version == ds.__version__ and ds.ADAM_OPTIMIZER == "adam" and callable(ds.replace_transformer_layer)
    assert ds.git_hash and ds.TORCH_DISTRIBUTED_DEFAULT_PORT == 29500 and ds.domino.__name__.endswith("domino")
    p = ds.add_tuning_arguments(argparse.ArgumentParser())
    args = p.parse_args(["--lr_schedule", "OneCycle", "--cycle_max_lr", "0.5"])
    cfg, err = L.get_config_from_args(args)
    assert err is None and cfg["type"] == "OneCycle"
    assert L.get_lr_from_config(cfg) == (0.5, "")
    assert L.get_lr_from_config({"type": "nope", "params": {}})[0] is None
    params = {}
    L.override_params(args, params)
    assert params[L.CYCLE_MAX_LR] == 0.5 and L.WARMUP_NUM_STEPS in params
    groups = [{"lr": 0.0}, {"lr": 0.0}]
    assert L.update_lr(groups, [0.1, 0.2]) == [0.1, 0.2]


def test_runtime_utils_helpers():
    from deepspeed_b200.runtime.utils import (DummyOptim, compare_tensors_in_structures, copy_to_device, get_flattened_grad_norm,
                                              get_weight_norm, is_moe_param, move_to_device, noop_context, offload_adam_states)
    from deepspeed_b200.runtime.zero.utils import apply_to_tensors_only, get_mapping_to_flat_buffer, isinstance_namedtuple
    w = torch.nn.Parameter(torch.tensor([3.0, 4.0]))
    assert DummyOptim([w]).param_groups[0]["params"][0] is w
    nested = {"a": [torch.ones(2), (torch.zeros(1), 5)], "b": "x"}
    moved = move_to_device(nested, "cpu")
    assert compare_tensors_in_structures(nested, moved) and moved["a"][1][1] == 5
    cp = copy_to_device(nested, "cpu")
    assert cp["a"][0] is not nested["a"][0] and compare_tensors_in_structures(cp, nested)
    assert not compare_tensors_in_structures(nested, {"a": [torch.ones(2)], "b": "x"})
    assert abs(float(get_weight_norm([w])) - 5.0) < 1e-6
    w.grad = torch.tensor([1.0, 2.0])
    assert abs(float(get_flattened_grad_norm([w], grad_norm_mask=[torch.tensor([[0, 1]])])) - 2.0) < 1e-6
    assert not is_moe_param(w)
    with noop_context():
        pass
    opt = torch.optim.Adam([w], lr=0.1)
    opt.step()
    offload_adam_states(opt, "cpu")
    assert opt.state[w]["exp_avg"].device.type == "cpu"
    from collections import namedtuple
    NT = namedtuple("NT", "x y")
    out = apply_to_tensors_only(lambda t: t + 1, NT(torch.zeros(1), [torch.ones(1), 7]))
    assert isinstance_namedtuple(out) and float(out.x) == 1.0 and float(out.y[0]) == 2.0 and out.y[1] == 7
    m = get_mapping_to_flat_buffer([torch.zeros(3), torch.zeros(2, 2)])
    assert [(o, n) for _, o, n in m] == [(0, 3), (3, 4)]


def test_logging_timer_group_and_fragment_names():
    from deepspeed_b200.checkpoint import SubparamShape
    from deepspeed_b200.module_inject import EmbeddingLayer, GroupQuantizer, Normalize
    from deepspeed_b200.runtime.config_utils import DeepSpeedConfigObject
    from deepspeed_b200.runtime.zero.config import read_zero_config_deprecated
    from deepspeed_b200.utils import groups, tensor_fragment
    from deepspeed_b200.utils.logging import get_current_level, should_log_le
    from deepspeed_b200.utils.tensor_fragment import fragment_address, map_to_flat_opt_states
    from deepspeed_b200.utils.timer import CudaEventTimer, mean
    assert should_log_le("critical") and get_current_level() >= 0 and mean([1, 3]) == 2 and CudaEventTimer is not None
    with pytest.raises(ValueError):
        should_log_le("loud")
    assert read_zero_config_deprecated({"zero_optimization": True, "allgather_size": 7}) == {"stage": 1, "allgather_bucket_size": 7}
    assert groups.get_model_parallel_world_size() == 1 and groups.get_tensor_model_parallel_src_rank() == 0
    groups.set_tensor_model_parallel_world_size(4)
    groups.set_tensor_model_parallel_rank(3)
    assert (groups.get_model_parallel_world_size(), groups.get_model_parallel_rank()) == (4, 3)
    groups.set_tensor_model_parallel_world_size(None)
    groups.set_tensor_model_parallel_rank(None)
    lp, hp = torch.zeros(4), torch.arange(10.)
    frag = tensor_fragment(lp_fragment=lp, lp_fragment_address=fragment_address(4, 0), hp_fragment=hp.narrow(0, 2, 4),
                           hp_fragment_address=fragment_address(4, 2))
    frag.update_lp()
    assert lp.tolist() == [2.0, 3.0, 4.0, 5.0]
    frag.set_optim_state_fragment(hp, {"exp_avg": torch.arange(10.) * 2, "step": torch.tensor(3)})
    assert frag.get_optim_state_fragment("exp_avg").tolist() == [4.0, 6.0, 8.0, 10.0] and frag.get_optim_state_keys() == ["exp_avg"]
    a, b = torch.nn.Parameter(torch.zeros(2)), torch.nn.Parameter(torch.zeros(3))
    state = {a: {"exp_avg": torch.ones(2)}, b: {"exp_avg": torch.full((3, ), 2.0)}}
    flat = torch.zeros(5)
    map_to_flat_opt_states(flat, [a, b], state, ["exp_avg"])
    assert state[flat]["exp_avg"].tolist() == [1, 1, 2, 2, 2] and state[b]["exp_avg"].data_ptr() == state[flat]["exp_avg"][2:].data_ptr()
    emb = EmbeddingLayer(weight=torch.nn.Parameter(torch.eye(4)))
    assert torch.equal(emb(torch.tensor([2])), torch.eye(4)[2:3])
    n = Normalize(dim=4, dtype=torch.float32)
    assert n(torch.randn(2, 4)).shape == (2, 4)
    q = GroupQuantizer(q_int8=True, group_size=4).quantize(torch.randn(16, 8))
    assert q.dtype == torch.int8 and q.scale.shape == (1, 4)
    assert SubparamShape(["a"], (4, 2), 0).partition_dim == 0

    class C(DeepSpeedConfigObject):

        def __init__(self):
            self.x = 1

    assert '"x": 1' in repr(C())


def _ds_ckpt_roundtrip(tmp):
    pytest.importorskip("transformers")
    from transformers import AutoConfig, AutoModelForCausalLM
    from deepspeed_b200.inference.v2 import build_engine_from_ds_checkpoint, build_hf_engine
    from deepspeed_b200.runtime.zero import unwrap_model_for_generation
    cfg = AutoConfig.for_model("llama", vocab_size=64, hidden_size=32, num_hidden_layers=1, num_attention_heads=4, num_key_value_heads=2,
                               intermediate_size=64, max_position_embeddings=64)
    torch.manual_seed(0)
    hf = AutoModelForCausalLM.from_config(cfg).eval()
    sm = {"state_manager": {"max_context": 64, "max_ragged_batch_size": 64, "max_ragged_sequence_count": 4,
                            "memory_config": {"mode": "allocate", "size": 8}}}
    eng = build_hf_engine(hf, sm, dtype=torch.float32, device="cpu")
    prompt = torch.randint(0, 64, (9, ))
    ref = eng.put([0], [prompt])[0]
    eng.serialize(tmp)
    eng2 = build_engine_from_ds_checkpoint(tmp, sm)
    out = eng2.put([0], [prompt])[0]
    assert torch.allclose(ref, out, atol=1e-6)
    import json
    import os
    from deepspeed_b200.inference.v2.model_implementations import flat_model_helpers as F
    assert os.path.exists(F.make_param_filename(tmp, 0, 1)) and os.path.exists(F.make_model_config_filename(tmp))
    md = F.ModelMetadata(**json.load(open(F.make_metadata_filename(tmp, 0, 1))))
    assert "0" in md.layers and "non_transformer" in md.layers and md.policy == "RaggedTransformer"
    emb = md.layers["non_transformer"].params["embed_w"].core_param
    assert emb.shape == (64, 32) and emb.strides == (32, 1) and emb.offset % 256 == 0
    with unwrap_model_for_generation(hf) as m:  # no ZeRO params: plain pass-through
        assert m is hf


def test_serialized_engine_roundtrip(tmp_path):
    run_distributed(_ds_ckpt_roundtrip, 1, (str(tmp_path), ))


def test_activation_checkpoint_functional_helpers():
    from deepspeed_b200.runtime.activation_checkpointing import checkpointing as C
    x = torch.randn(3, 4, requires_grad=True)
    d = C.detach_variable((x, 5))
    assert d[0].requires_grad and d[0].grad_fn is None and d[1] == 5
    t, o, f = C.extract_tensors((x, "a", torch.ones(1), 3))
    assert len(t) == 2 and o == ("a", 3) and f == (True, False, True, False)
    merged = C.merge_tensors(t, o, f)
    assert merged[1] == "a" and merged[2] is t[1]
    parts = C.partition_activations([x, 7])
    assert parts[1] == 7 and parts[0].numel() == 12  # tp = 1: the "partition" is the whole tensor
    packed = C.get_partitioned_activations_for_backward(parts, [x, 7])
    back = C.gather_partitioned_activations(packed)
    assert torch.equal(back[0], x.detach()) and back[1] == 7
    with pytest.raises(RuntimeError):
        C.detach_variable([x])


def test_functional_config_getters(tmp_path):
    from deepspeed_b200.compression import config as CC
    from deepspeed_b200.runtime import config as C
    from deepspeed_b200.runtime.data_pipeline import config as DC
    d = {"fp16": {"enabled": True, "loss_scale_window": 500, "initial_scale_power": 10},
         "optimizer": {"type": "AdamW", "params": {"lr": 1e-3, "max_grad_norm": 2.0}}, "scheduler": {"type": "WarmupLR", "params": {}},
         "train_batch_size": 8, "gradient_clipping": 1.5, "communication_data_type": "bf16",
         "sparse_attention": {"mode": "bigbird", "block": 32}, "eigenvalue": {"enabled": True, "max_iter": 7},
         "checkpoint": {"tag_validation": "fail", "parallel_write": {"pipeline_stage": True}}, "amp": {"enabled": True, "opt_level": "O1"}}
    assert C.get_fp16_enabled(d) and C.get_loss_scale(d) == 0 and C.get_initial_dynamic_scale(d) == 1024
    args = C.get_dynamic_loss_scale_args(d)
    assert args["scale_window"] == 500 and args["init_scale"] == 1024 and args["min_scale"] == 1
    assert C.get_optimizer_name(d) == "AdamW" and C.get_optimizer_gradient_clipping(d) == 2.0 and C.get_scheduler_name(d) == "WarmupLR"
    assert C.get_train_batch_size(d) == 8 and C.get_gradient_clipping(d) == 1.5 and C.get_communication_data_type(d) is torch.bfloat16
    assert C.get_amp_enabled(d) and C.get_amp_params(d) == {"opt_level": "O1"} and C.get_pld_enabled(d) is False
    sa = C.get_sparse_attention(d)
    assert sa["mode"] == "bigbird" and sa["block"] == 32 and sa["num_sliding_window_blocks"] == 3
    assert C.get_eigenvalue_config(d)[:3] == (True, False, 7) and C.get_eigenvalue_config({})[0] is False
    ck = C.get_checkpoint_params(d)
    assert C.get_checkpoint_tag_validation_mode(ck) == "FAIL" and C.get_checkpoint_parallel_write_pipeline(ck) is True
    with pytest.raises(C.DeepSpeedConfigError):
        C.get_checkpoint_tag_validation_mode({"tag_validation": "maybe"})
    with pytest.raises(ValueError):
        C.get_communication_data_type({"communication_data_type": "int3"})
    assert C.get_bfloat16_enabled({"bfloat16": {"enabled": True}}) and C.get_loss_scale({"bf16": {"enabled": True}}) == 1.0
    w = C.DeepSpeedConfigWriter()
    w.add_config("train_batch_size", 4)
    w.write_config(str(tmp_path / "c.json"))
    w2 = C.DeepSpeedConfigWriter()
    w2.load_config(str(tmp_path / "c.json"))
    assert w2.data == {"train_batch_size": 4}
    wq = CC.get_weight_quantization({"weight_quantization": {"shared_parameters": {"enabled": True},
                                                             "different_groups": {"g": {"params": {"start_bits": 8, "target_bits": 4}}}}})
    assert wq["shared_parameters"]["enabled"] and wq["different_groups"]["g"]["params"]["quantization_period"] == 1
    assert CC.get_layer_reduction_params({"layer_reduction": {"enabled": True, "keep_number_layer": 2}}) == {"keep_number_layer": 2}
    de = {"data_efficiency": {"enabled": True, "data_routing": {"random_ltd": {"enabled": True, "x": 1}}}}
    assert DC.get_data_efficiency_enabled(de) and DC.get_random_ltd_params(de) == {"x": 1} and DC.get_data_sampling_num_epochs(de) == 1000


def test_autotuning_utils_extra(tmp_path):
    from deepspeed_b200.autotuning import utils as U
    d = {"a": {"b": {"c": 3}}, "x": 1}
    assert U.get_val_by_key(d, "c") == 3 and U.get_val_by_key(d, "nope") is None
    U.set_val_by_key(d, "c", 9)
    assert d["a"]["b"]["c"] == 9
    hf = tmp_path / "hostfile"
    hf.write_text("worker-0 slots=8\n\n# comment\nworker-1 slots=4\n")
    assert list(U.fetch_hostfile(str(hf)).items()) == [("worker-0", 8), ("worker-1", 4)]
    assert U.fetch_hostfile(str(tmp_path / "missing")) is None
    assert U.validate_ds_config({"zero_optimization": {"stage": 1}})
    assert not U.validate_ds_config({"zero_optimization": {"stage": 2, "cpu_offload": True, "cpu_offload_params": True}})
    assert len(U.remove_dupe_dicts([{"a": 1, "b": 2}, {"b": 2, "a": 1}, {"a": 2}])) == 2
    assert U.prune_configs([{"a": 1, "z": {"k": 1}}, {"a": 1, "z": {"k": 2}}], ["z"]) == [{"a": 1}]
    assert U.get_tuning_keys({"a": [1, 2], "b": {"c": [1], "d": [3, 4]}}) == ["a", "d"]


def test_flops_profiler_module_helpers():
    import torch
    from deepspeed_b200.profiling.flops_profiler import profiler as P
    m = torch.nn.Sequential(torch.nn.Linear(8, 16), torch.nn.ReLU(), torch.nn.Linear(16, 4))
    prof = P.FlopsProfiler(m)
    prof.start_profile()
    calls = []
    f = P.wrapFunc(lambda x: x * 2, lambda x: (calls.append(1) or 100, 50))
    f(m(torch.randn(2, 8)))
    prof.stop_profile()
    assert P.get_module_flops(m) == prof.get_total_flops() and P.get_module_flops(m) >= 2 * 2 * (8 * 16 + 16 * 4) + 100
    assert P.get_module_macs(m[0]) == 2 * 8 * 16
    assert P.get_module_duration(m) >= 0 and calls == [1]
    prof.end_profile()


def test_env_report_helpers():
    from deepspeed_b200 import env_report as E
    assert E.human_readable_size(1536) == "1.50 KB"
    size, warns = E.get_shm_size()
    assert isinstance(size, str) and isinstance(warns, list)
    assert E.ninja_installed() in (True, False)


def test_model_parallel_region_ops_single_rank():
    import torch
    from deepspeed_b200.compression import basic_layer as B
    x = torch.randn(2, 8, requires_grad=True)
    for fn in (B.copy_to_model_parallel_region, B.reduce_from_model_parallel_region, B.scatter_to_model_parallel_region,
               B.gather_from_model_parallel_region):
        y = fn(x)
        y.sum().backward()
        assert torch.equal(y, x)
    a, b = B.split_tensor_along_last_dim(x, 2, contiguous_split_chunks=True)
    assert a.shape == (2, 4) and a.is_contiguous()


def test_op_builder_import_paths_and_probes():
    from deepspeed_b200.ops.op_builder import AsyncIOBuilder, FusedAdamBuilder  # noqa: F401
    from deepspeed_b200.ops.op_builder.cpu_adam import CPUAdamBuilder
    from deepspeed_b200.ops.op_builder.all_ops import __op_builders__
    from deepspeed_b200.op_builder import builder as B
    from deepspeed_b200.op_builder.fused_adam import FusedAdamBuilder as F2
    assert F2 is FusedAdamBuilder and len(__op_builders__) >= 20 and CPUAdamBuilder().is_compatible()
    assert B.get_default_compute_capabilities() == "10.0a" and B.TorchCPUOpBuilder is B.CPUOpBuilder
    b = B.CUDAOpBuilder()
    assert b.filter_ccs(["8.0", "9.0"]) == [["10", "0a"]] and b.simd_width().startswith("-D__")
    assert b.has_function("pthread_create", ("pthread", )) and not b.has_function("definitely_not_a_symbol_xyz", ("m", ))
    assert b.strip_empty_entries(["a", "", "b"]) == ["a", "b"] and b.builder() is b and not b.is_rocm_pytorch()


_NOT_PORTED = ("triton", "ccl.py", "hccl.py")  # tracing-compiler kernels and other vendors' collectives: out of scope by design
_ALLOWED_MISSING = {
    "env_report.py": set(),
    "runtime/zero/test.py": {"test1", "test2"},  # developer scratch file of the reference
    "module_inject/inject.py": {"test_hi"},  # ad-hoc demo function
}


def test_reference_public_names_exist_at_same_paths():
    """Every public top-level def/class of every upstream DeepSpeed module is importable from the same-path module here.
    The upstream names are stored in tests/golden/reference_public_names.json (regenerate:
    scripts/make_reference_golden.py)."""
    import importlib
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden",
                           "reference_public_names.json")) as fh:
        upstream = json.load(fh)
    assert len(upstream) > 100
    import deepspeed_b200
    mine = os.path.dirname(deepspeed_b200.__file__)
    problems = []
    for rel, names in upstream.items():
        if any(tag in rel for tag in _NOT_PORTED):
            continue
        want = set(names) - _ALLOWED_MISSING.get(rel, set())
        if not want:
            continue
        if not os.path.exists(os.path.join(mine, rel)):
            problems.append(f"{rel}: file missing ({sorted(want)[:4]}...)")
            continue
        modname = "deepspeed_b200." + rel[:-3].replace("/", ".")
        modname = modname[:-len(".__init__")] if modname.endswith(".__init__") else modname
        mod = importlib.import_module(modname)
        missing = sorted(n for n in want if not hasattr(mod, n))
        if missing:
            problems.append(f"{rel}: {missing}")
    assert not problems, "\n".join(problems)


def _engine_accessors():
    import torch
    import deepspeed_b200 as ds
    from deepspeed_b200.runtime import engine_accessors as A
    from deepspeed_b200.runtime.sparse_tensor import SparseTensor
    model = torch.nn.Linear(8, 8)
    eng, *_ = ds.initialize(model=model, config={"train_batch_size": 2, "optimizer": {"type": "Adam", "params": {"lr": 1e-3}},
                                                 "zero_optimization": {"stage": 1, "reduce_bucket_size": 1234},
                                                 "flops_profiler": {"enabled": False, "profile_step": 7},
                                                 "autotuning": {"enabled": False}})
    names = list(A._DIRECT) + [n for sec in A._NESTED.values() for n in sec]
    names += ["autotuning_enabled", "autotuning_metric_path", "autotuning_model_info_path", "autotuning_metric",
              "autotuning_profile_model_info", "flops_profiler_enabled", "flops_profiler_profile_step", "flops_profiler_detailed",
              "data_sampling_enabled", "curriculum_learning_enabled", "random_ltd_enabled", "zero_use_cpu_optimizer",
              "zero_cpu_offload", "zero_partial_offload", "zero_nvme_offload_optimizer", "postscale_gradients",
              "is_elastic_model_parallel_supported", "quantize_training", "get_pld_theta"]
    for n in names:
        getattr(eng, n)()  # every accessor resolves against a default config
    assert eng.zero_reduce_bucket_size() == 1234 and eng.flops_profiler_profile_step() == 7 and not eng.zero_cpu_offload()
    assert eng.autotuning_metric_path().endswith("autotuning_metric.json") and eng.postscale_gradients()
    assert eng.communication_data_type == torch.float32
    eng.communication_data_type = torch.bfloat16
    assert eng.communication_data_type == torch.bfloat16
    assert eng.is_map_style_dataset([1, 2]) and not eng.is_iterable_style_dataset([1])
    from deepspeed_b200 import comm as dist
    r = dist.get_rank()
    dense = torch.zeros(6, 4)
    dense[r] = r + 1.0
    dense[4] = 1.0
    sp = SparseTensor(dense)
    sp.orig_dense_tensor = dense
    want = torch.zeros(6, 4)
    want[0], want[1], want[4] = 0.5, 1.0, 1.0
    assert torch.allclose(eng.sparse_allreduce_bucket([sp], None)[0].to_dense(), want)
    eng.sparse_allreduce_no_retain([sp], None)
    assert torch.allclose(dense, want)
    ts = [torch.full((3, ), float(r + 1)), torch.full((2, 2), float(2 * r))]
    eng.allreduce_no_retain(ts, None, numel_per_bucket=2)
    assert torch.allclose(ts[0], torch.full((3, ), 1.5)) and torch.allclose(ts[1], torch.full((2, 2), 1.0))


def test_engine_config_accessors_and_sparse_collectives():
    run_distributed(_engine_accessors, 2)
