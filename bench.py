#!/usr/bin/env python
"""Headline benchmark: Llama-3-8B ZeRO-3 bf16 training throughput (tokens/s, whole job).

Contract (see task statement): ``python bench.py --gpus N --steps K --warmup W`` (N>1 is launched
under ``torch.distributed.run``).  W untimed warm-up steps, then exactly K timed steps bracketed by a
barrier + ``torch.cuda.synchronize()``; time is taken with CUDA events, max over ranks; rank 0 prints
ONE JSON line.  Two timed regions are measured back to back:

* ``value``      -- K steps of ``engine(ids, labels) / engine.backward / engine.step`` with the batch
                    already resident on the device (device-timed step throughput);
* ``e2e.value``  -- K steps through the same public API where every step first copies that step's
                    batch from pinned host memory (H2D) and reads the loss back to the host (D2H).

``--impl reference`` runs the UNMODIFIED reference DeepSpeed (installed under ``baseline/_ref``) with
an HF ``LlamaForCausalLM`` of the same architecture, ZeRO-3 bf16, its own FusedAdam -- same metric,
same config, same timing harness.

Synthetic data (random token ids of the benchmark shape) and random-init weights: there is no network
for datasets / checkpoints.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# same allocator setting for both arms: avoids fragmentation-induced OOMs near the 180 GB limit
os.environ.setdefault("PYTORCH_CUDA_ALLOC_CONF", "expandable_segments:True")


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--model", default="llama3-8b")
    ap.add_argument("--seq", type=int, default=4096)
    ap.add_argument("--micro-batch", type=int, default=2)
    ap.add_argument("--zero-stage", type=int, default=3)
    ap.add_argument("--layers", type=int, default=None, help="debug only: truncate depth (invalidates the result)")
    ap.add_argument("--checkpoint-layers", type=int, default=None)
    ap.add_argument("--fused-collectives", default="auto", choices=["auto", "on", "off"])
    ap.add_argument("--model-impl", default="native", choices=["native", "hf"],
                    help="b200 arm only: 'native' = deepspeed_b200.models.llama (fused kernels); 'hf' = the SAME "
                    "transformers.LlamaForCausalLM module the reference arm trains, under this framework's engine")
    ap.add_argument("--offload", default="none", choices=["none", "cpu"],
                    help="offload_optimizer device (both arms): fp32 master + Adam moments in pinned host memory, CPU Adam")
    ap.add_argument("--offload-ratio", type=float, default=1.0, help="Twin-Flow: fraction of the optimizer stepped on the host")
    ap.add_argument("--zero-init", action="store_true", help="construct the model under zero.Init (needed when the bf16 "
                    "parameters do not fit one GPU, e.g. llama3-70b)")
    ap.add_argument("--no-exposed", action="store_true", help="skip the 3 extra steps that measure exposed communication")
    ap.add_argument("--clip", type=float, default=0.0, help="gradient_clipping (both arms)")
    ap.add_argument("--gas", type=int, default=1, help="gradient_accumulation_steps (both arms); a timed step = one "
                    "optimizer step = GAS micro-batches")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="b200 arm: after the timed steps, write what the last timed step computed to DIR/<name>.npy")
    ap.add_argument("--local_rank", type=int, default=0)
    args = ap.parse_args()
    if args.dump_outputs and args.steps + args.warmup < 1:
        ap.error("--dump-outputs needs at least one step (--steps or --warmup) to take its outputs from")
    return args


def dump_outputs(torch, engine, losses, out_dir, rank, max_params=3, max_numel=1 << 26, sample=1 << 20):
    """What one training step hands its caller: the loss of each micro-batch, and the updated model.  The model is
    represented by the fp32 master weights of ``max_params`` weight matrices (first, middle and last of those with at
    most ``max_numel`` elements), each as a fixed seeded sample of ``sample`` elements; float32, about 12 MB in all.
    Collective under ZeRO-3: every rank calls it, rank 0 writes."""
    import numpy as np
    from deepspeed_b200.utils import safe_get_full_fp32_param
    arrays = {"loss": torch.stack([l.float().reshape(()) for l in losses]).cpu()}
    named = [(n, p) for n, p in engine.module.named_parameters()
             if len(getattr(p, "ds_shape", p.shape)) == 2 and int(getattr(p, "ds_numel", p.numel())) <= max_numel]
    picks = sorted({round(i * (len(named) - 1) / max(1, max_params - 1)) for i in range(max_params)}) if named else []
    for i in picks:
        name, p = named[i]
        full = safe_get_full_fp32_param(p).reshape(-1)
        if full.numel() > sample:
            idx = torch.randint(0, full.numel(), (sample, ), generator=torch.Generator().manual_seed(i))
            full = full[idx.to(full.device)]
        arrays[f"param.{name}"] = full.float().cpu()
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, f"{name}.npy"), a.numpy().astype(np.float32))


# ------------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, as prescribed by the profiling recipe)
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.idx)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_env(args):
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29500")
    os.environ.setdefault("RANK", str(rank))
    os.environ.setdefault("WORLD_SIZE", str(world))
    os.environ.setdefault("LOCAL_RANK", str(local))
    return rank, world, local


def host_memory_limit():
    """Bytes of host memory this process tree may use: min(MemAvailable, cgroup v2 / v1 limit)."""
    have = float("inf")
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                have = float(line.split()[1]) * 1024
    except OSError:
        pass
    for path in ("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory/memory.limit_in_bytes"):
        try:
            v = open(path).read().strip()
            if v.isdigit():
                have = min(have, float(v))
        except OSError:
            pass
    return have


def timed_loop(torch, dist_mod, world, steps, body):
    """barrier + sync, K steps under CUDA events, sync + barrier; returns max-over-ranks seconds."""
    if world > 1:
        dist_mod.barrier()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for i in range(steps):
        body(i)
    e.record()
    torch.cuda.synchronize()
    if world > 1:
        dist_mod.barrier()
    ms = torch.tensor([s.elapsed_time(e)], device="cuda", dtype=torch.float64)
    if world > 1:
        import torch.distributed as td
        td.all_reduce(ms, op=td.ReduceOp.MAX)
    return float(ms.item()) / 1e3


def common_config(args, world):
    """The part of the JSON line that must be IDENTICAL in both arms (the driver diffs it)."""
    par = f"zero{args.zero_stage}-dp{world}" + (f"-ep{world}" if args.model.startswith("mixtral") else "")
    return {
        "model": args.model + ("" if args.layers is None else f"-TRUNCATED-{args.layers}L"),
        "global_batch": args.micro_batch * world * args.gas,
        "micro_batch_per_gpu": args.micro_batch,
        "seq_len": args.seq,
        "parallelism": par,
        "zero_stage": args.zero_stage,
        "optimizer": "AdamW(lr=1e-5, betas=(0.9,0.95), eps=1e-8, wd=0.1), fp32 master + moments",
        "gradient_clipping": args.clip,
        "gradient_accumulation_steps": args.gas,
        "offload_optimizer": args.offload if args.offload == "none" else f"{args.offload} (ratio {args.offload_ratio})",
        "precision": "bf16 params/activations/grads-in-flight",
        "l2": "working set (>= 100 GB of parameter/optimizer state streamed per step) >> 126 MB L2",
    }


def ds_config_for(args, zero):
    if args.offload != "none":
        zero = dict(zero, offload_optimizer={"device": args.offload, "pin_memory": True, "ratio": args.offload_ratio})
    return {
        "train_micro_batch_size_per_gpu": args.micro_batch,
        "gradient_accumulation_steps": args.gas,
        "gradient_clipping": args.clip,
        "bf16": {"enabled": True},
        "optimizer": {"type": "AdamW", "params": {"lr": 1e-5, "betas": [0.9, 0.95], "eps": 1e-8, "weight_decay": 0.1}},
        "zero_optimization": zero,
        "steps_per_print": 10**9,
    }


def hf_llama(torch, mc, grad_ckpt=False):
    from transformers import LlamaConfig, LlamaForCausalLM
    hf_cfg = LlamaConfig(vocab_size=mc.vocab_size, hidden_size=mc.hidden_size, intermediate_size=mc.intermediate_size,
                         num_hidden_layers=mc.num_hidden_layers, num_attention_heads=mc.num_attention_heads,
                         num_key_value_heads=mc.num_key_value_heads, max_position_embeddings=mc.max_position_embeddings,
                         rms_norm_eps=mc.rms_norm_eps, rope_theta=mc.rope_theta, tie_word_embeddings=False,
                         use_cache=False)
    torch.manual_seed(1234)
    prev = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    with torch.device("cuda"):
        m = LlamaForCausalLM(hf_cfg)
    torch.set_default_dtype(prev)
    if grad_ckpt:
        m.gradient_checkpointing_enable()
    m.train()
    return m


def pick_checkpoint_layers(torch, cfg, micro_batch, seq, world, stage, explicit, offload=False):
    """Activation-recompute policy: keep everything when it fits in HBM, else checkpoint just enough
    layers.  Model states per rank (ZeRO-3): (2 + 4 + 4 + 4) B/param / world (+2 B/param gathered pool)."""
    if explicit is not None:
        return explicit
    free, total = torch.cuda.mem_get_info()
    n = cfg.num_parameters()
    per_param = 2 if offload else 14  # host offload leaves only the bf16 shard (+ transient gradient shards) on the device
    states = n * per_param / (world if stage >= 1 else 1) + (n * 2 if stage < 3 or world == 1 else 4 * 2 * 0.6e9)
    tokens = micro_batch * seq
    per_layer = tokens * cfg.hidden_size * 2 * 17.5 * 1.05  # ~17.5 h-sized bf16 tensors saved per layer
    ckpt_layer = tokens * cfg.hidden_size * 2 * 2.0
    fixed = 10e9 + tokens * cfg.hidden_size * 2 * 6
    budget = total * 0.94 - states - fixed
    L = cfg.num_hidden_layers
    k = 0
    while k < L and (L - k) * per_layer + k * ckpt_layer + per_layer > budget:
        k += 1
    return k


def run_b200(args):
    import torch
    rank, world, local = dist_env(args)
    torch.cuda.set_device(local)
    import deepspeed_b200 as ds
    from deepspeed_b200.models.llama import LlamaForCausalLM, llama_config
    from deepspeed_b200.ops import native
    native.cuda()
    ds.init_distributed(verbose=False)
    over = {}
    if args.layers is not None:
        over["num_hidden_layers"] = args.layers
    moe = args.model.startswith("mixtral") or args.model.endswith("-moe")
    if moe:
        # BASELINE config 3: Mixtral with expert parallelism over all ranks (dispatch / combine = the in-kernel NVLink
        # all-to-all of moe/symm_ep.py); dense parameters ZeRO-sharded over the data-parallel group
        from deepspeed_b200.models.mixtral import MixtralForCausalLM, mixtral_config
        cfg = mixtral_config(args.model, ep_size=world, **over)
        cfg.checkpoint_layers = 0
    else:
        cfg = llama_config(args.model, **over)
        cfg.checkpoint_layers = pick_checkpoint_layers(torch, cfg, args.micro_batch, args.seq, world, args.zero_stage,
                                                       args.checkpoint_layers, offload=args.offload != "none")
    hf = args.model_impl == "hf"
    zero = {"stage": args.zero_stage, "overlap_comm": True}
    if args.fused_collectives != "auto":
        zero["b200_fused_collectives"] = args.fused_collectives == "on"
    ds_config = ds_config_for(args, zero)
    hf_ckpt = bool(args.checkpoint_layers)
    if args.offload != "none":
        # host-offload sizing guard: fp32 master + two moments + fp32 gradient shard = 16 B/param of PINNED host memory for the
        # offloaded fraction, summed over the ranks of this node.  Refuse (cleanly) rather than take the box down.
        need = cfg.num_parameters() * 16.0 * args.offload_ratio + 8e9 * world
        have = host_memory_limit()
        if need > 0.85 * have:
            if rank == 0:
                print(json.dumps({"impl": "b200", "unavailable": f"host offload needs {need / 1e9:.0f} GB of pinned memory, "
                                  f"the box allows {have / 1e9:.0f} GB", "config": {"model": args.model, "n_gpus": world}}))
            return

    def build():
        if hf:
            # the engine's own contribution in isolation: same HF module as the reference arm, this framework's engine
            model = hf_llama(torch, cfg, grad_ckpt=hf_ckpt)
        else:
            torch.manual_seed(1234 + (rank if moe else 0))  # experts differ per rank, dense weights are broadcast
            prev = torch.get_default_dtype()
            torch.set_default_dtype(torch.bfloat16)
            if args.zero_init:
                # parameters are sharded as they are constructed: no rank ever holds the whole bf16 model
                with ds.zero.Init(config_dict_or_path=ds_config, dtype=torch.bfloat16):
                    model = LlamaForCausalLM(cfg)
            else:
                with torch.device("cuda"):
                    model = MixtralForCausalLM(cfg) if moe else LlamaForCausalLM(cfg)
            torch.set_default_dtype(prev)
        return ds.initialize(model=model, config=ds_config)[0]

    engine = build()
    B, S = args.micro_batch, args.seq
    g = torch.Generator().manual_seed(rank)
    n_batches = 4
    host = [torch.randint(0, cfg.vocab_size, (B, S), generator=g).pin_memory() for _ in range(n_batches)]
    dev = [h.cuda() for h in host]
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()

    gas = args.gas
    last_losses = [None] * gas  # the micro-batch losses of the latest step, for --dump-outputs

    def fwd(ids):
        return engine(input_ids=ids, labels=ids).loss if hf else engine(ids, labels=ids)

    def step_dev(i):
        for k in range(gas):
            loss = fwd(dev[(i * gas + k) % n_batches])
            engine.backward(loss)
            engine.step()
            last_losses[k] = loss.detach()

    def step_e2e(i):
        for k in range(gas):
            ids = host[(i * gas + k) % n_batches].to("cuda", non_blocking=True)  # H2D from pinned memory, every micro step
            loss = fwd(ids)
            engine.backward(loss)
            engine.step()
            last_losses[k] = loss.detach()
        loss_host.copy_(loss.detach().float().reshape(1), non_blocking=False)  # D2H read of the result

    try:
        for i in range(args.warmup):
            step_e2e(i)
    except torch.OutOfMemoryError:
        if not hf or hf_ckpt:
            raise
        # same policy as the reference arm: the HF module keeps every activation; retry with HF gradient checkpointing
        engine.destroy() if hasattr(engine, "destroy") else None
        del engine
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        hf_ckpt = True
        engine = build()
        for i in range(args.warmup):
            step_e2e(i)
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
    l0 = native.launch_count
    t_dev = timed_loop(torch, ds.comm, world, args.steps, step_dev)
    launches = native.launch_count - l0
    t_e2e = timed_loop(torch, ds.comm, world, args.steps, step_e2e)
    clocks = sampler.stop() if rank == 0 else None
    if args.dump_outputs:
        dump_outputs(torch, engine, last_losses, args.dump_outputs, rank)
    # exposed (non-overlapped) communication: 2 extra, untimed-for-throughput steps with every compute-stream
    # wait on a collective bracketed by CUDA events (the bracket holds no kernels => elapsed == stall)
    exposed = None
    if world > 1 and hasattr(engine.optimizer, "measure_exposed") and not args.no_exposed:
        step_dev(0)  # settle: absorbs the rank skew left by the timing epilogue (host-side all-reduce of the timings)
        torch.cuda.synchronize()
        ds.comm.barrier()
        engine.optimizer.measure_exposed(True)
        for i in range(2):
            step_dev(i)
        ex = engine.optimizer.exposed_ms()
        engine.optimizer.measure_exposed(False)
        t = torch.tensor([ex["all_gather"] / 2, ex["reduce"] / 2], device="cuda")
        ds.comm.all_reduce(t, op=ds.comm.ReduceOp.MAX)
        exposed = {"all_gather_ms_per_step": float(t[0]), "reduce_scatter_adam_ms_per_step": float(t[1]),
                   "total_ms_per_step": float(t[0] + t[1]), "how": "CUDA-event brackets around compute-stream waits, "
                   "max over ranks, mean of 2 steps"}
    tokens_per_step = B * S * world * gas
    if rank == 0:
        val = tokens_per_step * args.steps / t_dev
        e2e = tokens_per_step * args.steps / t_e2e
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        if moe:  # active parameters per token: attention + top-k experts + router
            h_, i_, L_ = cfg.hidden_size, cfg.intermediate_size, cfg.num_hidden_layers
            mm = 2 * (h_ * (cfg.q_size + 2 * cfg.kv_size) + cfg.q_size * h_ + cfg.num_experts_per_tok * 3 * h_ * i_ +
                      h_ * cfg.num_local_experts) * L_ + 2 * h_ * cfg.vocab_size
            flops = 3 * (mm + 4 * S * cfg.q_size * L_ * 0.5) * val / world
        else:
            flops = cfg.flops_per_token(S) * val / world
        out = {
            "metric": ("tokens/sec (whole job, device-timed, max over ranks) Llama-3-8B ZeRO-3 bf16 training"
                       if (args.model == "llama3-8b" and args.zero_stage == 3) else
                       f"tokens/sec (whole job, device-timed, max over ranks) {args.model} ZeRO-{args.zero_stage} bf16 training"),
            "value": val,
            "unit": "tokens/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": t_dev / args.steps * 1e3,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "bf16",
            "data": "synthetic random token ids, random-init weights (no network for datasets/checkpoints)",
            "impl": "b200",
            "config": common_config(args, world),
            "details": {
                "model_impl": "transformers.LlamaForCausalLM (sdpa)" if hf else "deepspeed_b200.models.llama (fused sm_100a kernels)",
                "optimizer_impl": "fused sm_100a AdamW kernel",
                "activation_checkpoint_layers": cfg.checkpoint_layers if not hf else None,
                "hf_gradient_checkpointing": hf_ckpt if hf else None,
                "fused_in_backward_optimizer": bool(engine.optimizer.fused_in_backward),
                "collectives": "nvlink-peer-kernels" if engine.optimizer._symm is not None else "nccl",
                "gemm_backend": __import__("deepspeed_b200.ops.gemm", fromlist=["x"]).get_backend(),
                "gemm_choices": _gemm_choice_summary(),
            },
            "model_tflops_per_gpu": flops / 1e12,
            "mfu_vs_measured_sustained": (flops / 1e12) / peaks["bf16_tflops_sustained"] if peaks.get(
                "bf16_tflops_sustained") else None,
            "clocks": clocks,
            "e2e": {
                "value": e2e,
                "unit": "tokens/s",
                "ms_per_step": t_e2e / args.steps * 1e3,
                "h2d_bytes_per_step": B * S * 8 * gas,
                "d2h_bytes_per_step": 4,
            },
            "gpu_launches": launches,
            "max_mem_gb": torch.cuda.max_memory_allocated() / 2**30,
            "exposed_comm": exposed,
        }
        print(json.dumps(out), flush=True)


def _gemm_choice_summary():
    """Which implementation served each distinct GEMM problem of the step (persisted table / first-use measurement)."""
    from deepspeed_b200.ops import gemm
    used = gemm.tuning_table()
    own = sorted(k for k, v in used.items() if v == "own")
    lib = sorted(k for k, v in used.items() if v == "lib")
    return {"own_tcgen05": len(own), "cublas": len(lib), "cublas_shapes": lib, "measured_online": gemm.tuning_measurements()}


def run_reference(args):
    rank, world, local = dist_env(args)
    ref_dir = os.path.join(ROOT, "baseline", "_ref")
    if not os.path.isdir(os.path.join(ref_dir, "deepspeed")):
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": "baseline/_ref/deepspeed is not installed"}))
        return
    sys.path.insert(0, ref_dir)
    os.environ.setdefault("TORCH_EXTENSIONS_DIR", os.path.join(ref_dir, "_torch_extensions"))
    os.environ.setdefault("TORCH_CUDA_ARCH_LIST", "10.0")
    os.environ.setdefault("DS_SKIP_CUDA_CHECK", "1")
    try:
        import torch
        torch.cuda.set_device(local)
        import deepspeed  # the unmodified reference
        from transformers import LlamaConfig, LlamaForCausalLM
    except Exception as e:  # pragma: no cover
        if rank == 0:
            print(json.dumps({"impl": "reference", "unavailable": f"import failed: {e!r}"[:300]}))
        return
    sys.path.insert(0, ROOT)
    from deepspeed_b200.models.llama import llama_config
    over = {}
    if args.layers is not None:
        over["num_hidden_layers"] = args.layers
    mc = llama_config(args.model, **over)
    deepspeed.init_distributed(dist_backend="nccl")
    B, S = args.micro_batch, args.seq
    ds_config = ds_config_for(args, {"stage": args.zero_stage, "overlap_comm": True})

    def build(grad_ckpt):
        m = hf_llama(torch, mc, grad_ckpt)
        eng, _, _, _ = deepspeed.initialize(model=m, model_parameters=m.parameters(), config=ds_config)
        return eng

    g = torch.Generator().manual_seed(rank)
    n_batches = 4
    host = [torch.randint(0, mc.vocab_size, (B, S), generator=g).pin_memory() for _ in range(n_batches)]
    loss_host = torch.zeros(1, dtype=torch.float32).pin_memory()
    ckpt_used = args.checkpoint_layers is not None and args.checkpoint_layers > 0
    engine = None
    for attempt in range(2):
        try:
            engine = build(ckpt_used)
            dev = [h.cuda() for h in host]

            gas = args.gas

            def step_dev(i):
                for k in range(gas):
                    ids = dev[(i * gas + k) % n_batches]
                    loss = engine(input_ids=ids, labels=ids).loss
                    engine.backward(loss)
                    engine.step()

            def step_e2e(i):
                for k in range(gas):
                    ids = host[(i * gas + k) % n_batches].to("cuda", non_blocking=True)
                    loss = engine(input_ids=ids, labels=ids).loss
                    engine.backward(loss)
                    engine.step()
                loss_host.copy_(loss.detach().float().reshape(1))

            for i in range(args.warmup):
                step_e2e(i)
            break
        except torch.OutOfMemoryError:
            if ckpt_used:
                if rank == 0:
                    print(json.dumps({"impl": "reference", "unavailable": "CUDA OOM even with HF gradient checkpointing"}))
                return
            del engine
            engine = None
            import gc
            gc.collect()
            torch.cuda.empty_cache()
            ckpt_used = True
    sampler = ClockSampler(torch.cuda.current_device())
    if rank == 0:
        sampler.start()
    import torch.distributed as td

    class _D:
        barrier = staticmethod(td.barrier)

    t_dev = timed_loop(torch, _D, world, args.steps, step_dev)
    t_e2e = timed_loop(torch, _D, world, args.steps, step_e2e)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        tokens_per_step = B * S * world * args.gas
        out = {
            "metric": "tokens/sec (whole job, device-timed, max over ranks) Llama-3-8B ZeRO-3 bf16 training",
            "value": tokens_per_step * args.steps / t_dev,
            "unit": "tokens/s",
            "n_gpus": world,
            "steps": args.steps,
            "warmup": args.warmup,
            "ms_per_step": t_dev / args.steps * 1e3,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": "bf16",
            "data": "synthetic random token ids, random-init weights",
            "impl": "reference",
            "config": common_config(args, world),
            "details": {
                "model_impl": "transformers.LlamaForCausalLM (sdpa)",
                "optimizer_impl": "reference FusedAdam (AdamW)",
                "hf_gradient_checkpointing": ckpt_used,
                "deepspeed_version": deepspeed.__version__,
            },
            "clocks": clocks,
            "e2e": {"value": tokens_per_step * args.steps / t_e2e, "unit": "tokens/s",
                    "ms_per_step": t_e2e / args.steps * 1e3, "h2d_bytes_per_step": B * S * 8 * args.gas,
                    "d2h_bytes_per_step": 4},
            "gpu_launches": 0,
            "max_mem_gb": torch.cuda.max_memory_allocated() / 2**30,
        }
        print(json.dumps(out), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        try:
            run_reference(args)
        except Exception as e:  # the contract: print an 'unavailable' line and exit 0
            if int(os.environ.get("RANK", 0)) == 0:
                import traceback
                traceback.print_exc()
                print(json.dumps({"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"[:300]}))
        return
    run_b200(args)


if __name__ == "__main__":
    main()
