#!/usr/bin/env python
"""Regenerate the upstream-DeepSpeed fixtures under ``tests/golden/`` that the interop tests compare against.

    python scripts/make_reference_golden.py /path/to/DeepSpeed      # an upstream source checkout

Runs upstream DeepSpeed on the CPU (gloo, two ranks) and stores only data: the public names of its modules, index
files its ``indexed_dataset`` writes, checkpoints its engine saves, and the weights its ``zero_to_fp32.py`` consolidates
from checkpoints this project saves.  No upstream source is copied.
"""
import ast
import glob
import importlib.util
import json
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, ROOT)


def public_names(ref):
    """{module path relative to the package: sorted public top-level defs / classes} of upstream's ``deepspeed``."""
    pkg = os.path.join(ref, "deepspeed")
    out = {}
    for root, _, files in os.walk(pkg):
        for f in files:
            if not f.endswith(".py"):
                continue
            path = os.path.join(root, f)
            try:
                tree = ast.parse(open(path).read())
            except SyntaxError:
                continue
            names = sorted(n.name for n in tree.body
                           if isinstance(n, (ast.FunctionDef, ast.ClassDef)) and not n.name.startswith("_"))
            if names:
                out[os.path.relpath(path, pkg)] = names
    with open(os.path.join(GOLDEN, "reference_public_names.json"), "w") as fh:
        json.dump(dict(sorted(out.items())), fh, indent=0, sort_keys=True)


def indexed_datasets(ref):
    """The samples of ``test_indexed_dataset_formats_and_interop`` written by upstream's builders."""
    f = os.path.join(ref, "deepspeed", "runtime", "data_pipeline", "data_sampling", "indexed_dataset.py")
    spec = importlib.util.spec_from_file_location("_upstream_indexed_dataset", f)
    R = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(R)
    samples = [np.arange(5), np.arange(3) + 10, np.arange(7) + 100]
    out = os.path.join(GOLDEN, "indexed_dataset")
    os.makedirs(out, exist_ok=True)
    for name, builder in (("mmap_int32", lambda p: R.MMapIndexedDatasetBuilder(R.data_file_path(p), dtype=np.int32)),
                          ("mmap_uint16", lambda p: R.MMapIndexedDatasetBuilder(R.data_file_path(p), dtype=np.uint16)),
                          ("legacy_int32", lambda p: R.IndexedDatasetBuilder(R.data_file_path(p), dtype=np.int32))):
        prefix = os.path.join(out, name)
        b = builder(prefix)
        for s in samples:
            b.add_item(torch.from_numpy(s))
            b.end_document()
        b.finalize(R.index_file_path(prefix))


def _torchrun(script, args, env):
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", "29731", script] + args, env=env,
                       capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]


def upstream_checkpoints(ref):
    """Upstream trains 3 steps, saves (tag ``ref3``), trains 2 more and records the parameters (``expect_after5.pt``)."""
    from tests.unit.test_checkpoint_cpu import _REF_SAVE
    env = dict(os.environ, DS_ACCELERATOR="cpu", PYTHONPATH=ROOT, PYTHONDONTWRITEBYTECODE="1")
    with tempfile.TemporaryDirectory() as tmp:
        script = os.path.join(tmp, "ref_save.py")
        with open(script, "w") as fh:
            fh.write(_REF_SAVE.format(ref=ref, root=ROOT))
        for stage in (2, 3):
            out = os.path.join(GOLDEN, f"ref_ckpt_stage{stage}")
            shutil.rmtree(out, ignore_errors=True)
            os.makedirs(out)
            _torchrun(script, [out, str(stage)], env)
            for f in glob.glob(os.path.join(out, "**", "*.py"), recursive=True):
                os.remove(f)  # upstream copies its zero_to_fp32.py next to every checkpoint


def upstream_consolidation(ref):
    """Checkpoints saved here (``_save_worker``), consolidated by upstream's ``zero_to_fp32.py``; stores the checkpoint
    files upstream read (``t3/*.pt``) and the weights it produced (``consolidated.pt``)."""
    from tests.common import run_distributed
    from tests.unit.test_checkpoint_cpu import _save_worker
    env = dict(os.environ, PYTHONPATH=ref, DS_ACCELERATOR="cpu", PYTHONDONTWRITEBYTECODE="1")
    for stage in (1, 3):
        with tempfile.TemporaryDirectory() as d:
            run_distributed(_save_worker, 2, (d, stage))
            cons = os.path.join(d, "consolidated")
            # run from the checkpoint directory, as upstream does: inside its package, utils/logging.py shadows the stdlib
            script = os.path.join(d, "stock_zero_to_fp32.py")
            shutil.copyfile(os.path.join(ref, "deepspeed", "utils", "zero_to_fp32.py"), script)
            p = subprocess.run([sys.executable, script, d, cons, "--tag", "t3"], env=env, capture_output=True, text=True,
                               timeout=900, cwd=d)
            assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
            got = {}
            for f in sorted(os.listdir(cons)):
                if f.endswith(".bin") or f.endswith(".pt"):
                    got.update(torch.load(os.path.join(cons, f), map_location="cpu", weights_only=False))
            assert got, os.listdir(cons)
            out = os.path.join(GOLDEN, f"zero_to_fp32_stage{stage}")
            shutil.rmtree(out, ignore_errors=True)
            os.makedirs(os.path.join(out, "t3"))
            torch.save({k: v.float().clone() for k, v in got.items()}, os.path.join(out, "consolidated.pt"))
            for f in sorted(os.listdir(os.path.join(d, "t3"))):
                if f.endswith(".pt"):
                    shutil.copyfile(os.path.join(d, "t3", f), os.path.join(out, "t3", f))


if __name__ == "__main__":
    ref = os.path.abspath(sys.argv[1])
    os.makedirs(GOLDEN, exist_ok=True)
    public_names(ref)
    indexed_datasets(ref)
    upstream_checkpoints(ref)
    upstream_consolidation(ref)
