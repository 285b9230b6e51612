"""bench.py --dump-outputs: what it writes is the step's output, exactly, in float arrays under 64 MB."""
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
import bench  # noqa: E402


def _load(d):
    return {f.stem: np.load(f) for f in sorted(Path(d).glob("*.npy"))}


def test_dump_is_exact_for_every_group_of_a_small_step(tmp_path):
    n, P, L, ds = 3000, 2, 1366, 1376
    g = torch.Generator().manual_seed(7)
    parity = torch.randint(0, 256, (P, n, ds), dtype=torch.uint8, generator=g)
    committed = torch.randint(-(1 << 63), (1 << 63) - 1, (n,), dtype=torch.int64, generator=g)
    bar = torch.randint(0, 65, (n,), dtype=torch.int32, generator=g)
    bench.dump_step_outputs(torch, "cpu", tmp_path, parity, committed, bar, n, L)
    out = _load(tmp_path)
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert (out["groups"] == np.arange(n)).all()
    assert (out["parity"] == parity[:, :, :L].numpy()).all()
    cw = out["commit_words"].astype(np.uint64)
    assert ((cw[:, 0] | (cw[:, 1] << np.uint64(32))) == committed.numpy().view(np.uint64)).all()
    assert (out["commit_bar"] == bar.numpy()).all()


def test_dump_of_a_full_step_is_a_fixed_sample_under_64_mb(tmp_path):
    n, P, L, ds = 1 << 20, 2, 1366, 1376
    rows = torch.randint(0, 256, (P, 1, ds), dtype=torch.uint8)
    parity = rows.expand(P, n, ds)
    committed = torch.arange(n, dtype=torch.int64)
    bar = (torch.arange(n, dtype=torch.int32) % 65)
    sizes = []
    for run in ("a", "b"):
        bench.dump_step_outputs(torch, "cpu", tmp_path / run, parity, committed, bar, n, L)
        sizes.append(sum(f.stat().st_size for f in (tmp_path / run).glob("*.npy")))
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert max(sizes) <= 64_000_000
    assert all((a[k] == b[k]).all() for k in a)
    idx = a["groups"].astype(np.int64)
    assert 1000 < len(idx) < n and (np.diff(idx) > 0).all()
    assert (a["commit_words"][:, 0] == idx).all() and (a["commit_bar"] == idx % 65).all()
    assert (a["parity"] == rows[:, :, :L].numpy()).all()
