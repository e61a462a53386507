"""bench.py --dump-outputs: what the last timed step returned, written as .npy files so that two builds can be compared
output for output.  CPU: the size budget and the seeded sampling of oversized arrays.  GPU: two runs with the same
arguments write the same arrays (the gradients up to the order of the kernels' atomic additions)."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest
import torch

from _util import small_config
from multi_modal_foundation_model_b200.model import build_model

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class _Store:
    """Stand-in for the engine's ParamStore: every gradient is 0, 1, 2, ... so a sample shows where it came from."""

    def __init__(self, model):
        self.grads = {n: torch.arange(p.numel(), dtype=torch.float32).view(p.shape) for n, p in model.named_parameters()}

    def g(self, name):
        return self.grads[name]


def test_dump_outputs_budget_and_sampling(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 256 << 10)
    model = build_model(16, 2, small_config())
    store = _Store(model)
    preds = {"ap": torch.arange(4 * 100 * 16, dtype=torch.float32).view(4, 100, 16),
             "behavior": torch.arange(4 * 100 * 2, dtype=torch.float32).view(4, 100, 2)}
    out = types.SimpleNamespace(loss=torch.tensor(1.5), mod_loss={m: torch.tensor(0.5) for m in preds},
                                mod_n_examples={m: torch.tensor(7) for m in preds}, mod_preds=preds)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), out, model, store)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    assert len(files) == 1 + 3 * len(preds) + len(list(model.parameters()))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 256 << 10
    full = {f"{k}.npy": v for k, v in [("loss", out.loss)] + [(f"mod_preds.{m}", v) for m, v in preds.items()]
            + [(f"grad.{n}", g) for n, g in store.grads.items()]}
    n_sampled = 0
    for f in files:
        x = np.load(tmp_path / "a" / f)
        assert np.array_equal(x, np.load(tmp_path / "b" / f)), f               # the same positions in every run
        if f.startswith("mod_n_examples."):
            assert x.dtype == np.float64 and x == 7
            continue
        assert x.dtype == np.float32
        ref = full.get(f)
        if ref is not None and x.shape != tuple(ref.shape):
            # a sample: 1-D, distinct flat positions in increasing order (the values are the positions here)
            n_sampled += 1
            assert x.ndim == 1 and 0 < x.size < ref.numel() and (np.diff(x) > 0).all(), f
            assert np.isin(x, ref.flatten().numpy()).all(), f
        elif ref is not None:
            assert np.array_equal(x, ref.numpy()), f
    assert n_sampled > 0 and np.load(tmp_path / "a" / "loss.npy") == np.float32(1.5)


def _bench(out_dir):
    args = ["--gpus", "1", "--steps", "2", "--warmup", "3", "--no-cpu-baseline", "--no-library-bar",
            "--sustained-seconds", "0", "--dump-outputs", str(out_dir)]
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_dump_outputs_repeat_across_runs(tmp_path):
    la, lb = _bench(tmp_path / "a"), _bench(tmp_path / "b")
    assert la["steps"] == lb["steps"] == 2
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(os.listdir(tmp_path / "b"))
    assert {"loss.npy", "mod_preds.ap.npy", "mod_preds.behavior.npy", "grad.decoder_norm.weight.npy"} <= set(files)
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= 64 * 10 ** 6
    for f in files:
        x, y = np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f)
        assert x.dtype in (np.float32, np.float64) and x.shape == y.shape and np.isfinite(x).all(), f
        if f.startswith("mod_n_examples."):
            assert np.array_equal(x, y), f
        else:
            x, y = x.astype(np.float64), y.astype(np.float64)
            assert np.linalg.norm(x - y) <= 1e-4 * np.linalg.norm(y) + 1e-12, f
