"""bench.dump_outputs on host tensors: exact float32 / float64 copies of every output, and a fixed seeded sample of the boards when
they do not fit in the size limit."""
import importlib.util
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _outputs(B):
    g = torch.Generator().manual_seed(0)
    return {"priors": torch.rand((B, 209), generator=g), "value": torch.rand((B,), generator=g) * 2 - 1,
            "mask": torch.randint(-2 ** 31, 2 ** 31 - 1, (B, 8), dtype=torch.int32, generator=g),
            "pawn": torch.randint(0, 256, (B, 8), dtype=torch.int32, generator=g).to(torch.uint8)}


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_is_exact_and_sampled_under_the_limit(tmp_path, monkeypatch):
    bench = _bench()
    outs = _outputs(300)
    bench.dump_outputs(str(tmp_path / "all"), outs)
    got = _load(tmp_path / "all")
    assert sorted(got) == ["board_index", "mask", "pawn", "priors", "value"]
    assert all(v.dtype in (np.float32, np.float64) for v in got.values())
    assert np.array_equal(got["board_index"], np.arange(300))
    assert np.array_equal(got["priors"], outs["priors"].numpy()) and np.array_equal(got["value"], outs["value"].numpy())
    assert np.array_equal(got["mask"].astype(np.uint32), outs["mask"].numpy().view(np.uint32))
    assert np.array_equal(got["pawn"], outs["pawn"].numpy())

    limit = 4096 + 100 * 944   # room for 100 boards of 836 + 4 + 64 + 32 bytes and their index
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", limit)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), outs)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit
    idx = a["board_index"].astype(np.int64)
    assert len(idx) == 100 and np.all(np.diff(idx) > 0) and idx[-1] < 300
    assert all(np.array_equal(a[k], b[k]) for k in a)                # the same sample every run
    assert np.array_equal(a["priors"], outs["priors"].numpy()[idx]) and np.array_equal(a["mask"], got["mask"][idx])
