"""bench.py --dump-outputs: the outputs of the last timed step as float32 / float64 .npy files, exact, and within the size
cap through the same seeded sample of items on every run."""
import json
import pathlib
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = pathlib.Path(__file__).resolve().parent.parent


def _load(d):
    return {p.stem: np.load(p) for p in d.glob("*.npy")}


def test_dump_outputs_exact_and_sampled_under_the_cap(tmp_path, monkeypatch):
    n = 1000
    verdicts = (np.arange(n) % 3).astype(np.uint8)
    values = np.arange(n, dtype=np.uint64) << 40
    tally = np.arange(5 * 64, dtype=np.uint8).reshape(5, 64)
    names, arrays = ("verdicts", "values", "tally"), [verdicts, values, tally]
    bench.dump_outputs(tmp_path / "all", names, arrays, n)
    got = _load(tmp_path / "all")
    assert set(got) == set(names)
    assert got["verdicts"].dtype == got["tally"].dtype == np.float32 and got["values"].dtype == np.float64
    assert (got["verdicts"] == verdicts).all() and (got["values"] == values).all() and (got["tally"] == tally).all()

    cap = 4096 + tally.size * 4 + 100 * (4 + 8 + 8)       # room for 100 items
    monkeypatch.setattr(bench, "DUMP_BYTES", cap)
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, names, arrays, n)
        assert sum(p.stat().st_size for p in (tmp_path / d).glob("*.npy")) <= cap
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert set(a) == set(names) | {"sample_index"} and all((a[k] == b[k]).all() for k in a)
    idx = a["sample_index"].astype(np.int64)
    assert len(idx) == 100 and len(set(idx.tolist())) == 100 and (np.diff(idx) > 0).all()
    assert (a["verdicts"] == verdicts[idx]).all() and (a["values"] == values[idx]).all() and (a["tally"] == tally).all()


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path(tmp_path):
    import oracle as O
    out = tmp_path / "out"
    n, unique = 5000, 257
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--config", "2", "--items", str(n), "--unique", str(unique),
                          "--steps", "2", "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)],
                         stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900, cwd=str(ROOT))
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout)["steps"] == 2
    got = _load(out)
    assert set(got) == {"verdicts", "tally"}
    wl = bench.Choice()
    wl.make(unique, 0)
    cts, rings, sums = (bench.tile(a, n) for a in wl.inputs)
    ov, ot = O.verify_choice_batch(wl.pk, 5, True, cts, rings, sums)
    assert got["verdicts"].dtype == np.float32 and (got["verdicts"] == ov).all()
    assert got["tally"].shape == (5, 64) and (got["tally"] == ot).all()
