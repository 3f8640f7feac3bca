"""Host logic of bench.py: the headline times exactly --steps iterations (default per workload), and --dump-outputs
writes the same bounded sample in every run, gathered correctly from the shards."""
import json
import os
import sys

import numpy as np
import pytest

import bench
from lbfgsb_b200 import sharded


def _parse(args, monkeypatch):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + args)
    return bench.parse()


def test_steps_default_per_workload_and_bad_arguments(monkeypatch):
    assert _parse([], monkeypatch).steps == 20
    assert _parse(["--workload", "quadratic"], monkeypatch).steps == 12
    assert _parse(["--workload", "driver3_f32"], monkeypatch).steps == 20
    a = _parse(["--gpus", "1", "--steps", "7", "--warmup", "3", "--dump-outputs", "out"], monkeypatch)
    assert (a.steps, a.warmup, a.dump_outputs) == (7, 3, "out")
    for bad in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]):
        with pytest.raises(SystemExit):
            _parse(bad, monkeypatch)


class _Head(dict):
    def __missing__(self, key):
        return 0


@pytest.mark.parametrize("args,k", [([], 20), (["--steps", "7"], 7), (["--workload", "quadratic"], 12),
                                    (["--workload", "quadratic", "--steps", "20"], 20)])
def test_main_times_the_requested_steps(args, k, monkeypatch, capfd):
    """The K that main() hands to the headline and to the e2e arm, with the device work stubbed out."""
    seen = {}

    class Ctx:
        world, rank, comm = 1, 0, None

    def measure(cx, kind, n_global, m, dtype, l_odd, W, K, *a, **kw):
        seen["measure"] = K
        return _Head(value=1.0)

    def e2e_host(cx, kind, n_global, m, W, K, l_odd):
        seen["e2e"] = K
        return {}

    monkeypatch.setattr(bench, "Ctx", Ctx)
    monkeypatch.setattr(bench, "measure", measure)
    monkeypatch.setattr(bench, "e2e_host", e2e_host)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--no-extra", "--no-cpu"] + args)
    bench.main()
    assert seen == {"measure": k, "e2e": k}
    assert json.loads(capfd.readouterr().out.strip().splitlines()[-1])["steps"] == k


@pytest.mark.parametrize("n", [1, 1000, bench.DUMP_SAMPLE, bench.DUMP_SAMPLE + 1, 100_000_000, 400_000_000])
def test_dump_index_is_one_per_stretch_and_bounded(n):
    idx = bench.dump_index(n)
    size = min(n, bench.DUMP_SAMPLE)
    assert idx.dtype == np.int64 and idx.size == size
    edge = np.arange(size + 1, dtype=np.int64) * n // size
    assert np.all(idx >= edge[:-1]) and np.all(idx < edge[1:])
    if n <= bench.DUMP_SAMPLE:
        assert np.array_equal(idx, np.arange(n))


def test_dump_index_is_pinned():
    """Integer arithmetic only: these values hold in every run and with every numpy version."""
    idx = bench.dump_index(100_000_000)
    assert idx[:4].tolist() == [13, 98, 272, 375] and int(idx[-1]) == 99999952
    assert bench.dump_index(125_000_000)[:4].tolist() == [69, 142, 347, 396]


@pytest.mark.parametrize("world", [1, 2, 3, 8])
def test_shards_together_give_every_sampled_value_once(world):
    n_global = 10007
    idx = bench.dump_index(n_global, 1000)
    v = np.random.default_rng(1).standard_normal(n_global)
    merged = np.zeros(idx.size)
    hits = np.zeros(idx.size, np.int64)
    for rank in range(world):
        lo, hi = sharded.shard_bounds(n_global, rank, world)
        dst, src = bench.shard_positions(idx, lo, hi)
        part = np.zeros(idx.size)
        part[dst] = v[lo:hi][src]
        merged += part
        hits[dst] += 1
    assert np.all(hits == 1)
    assert np.array_equal(merged, v[idx])


def test_written_outputs_round_trip_within_64_mib(tmp_path):
    idx = bench.dump_index(100_000_000)
    outputs = {"x": np.sqrt(idx + 1.0), "g": -np.sqrt(idx + 2.0), "f": np.array([1.5]), "index": idx.astype(np.float64)}
    d = os.path.join(str(tmp_path), "out")
    bench.write_outputs(d, outputs)
    assert sorted(os.listdir(d)) == ["f.npy", "g.npy", "index.npy", "x.npy"]
    assert sum(os.path.getsize(os.path.join(d, f)) for f in os.listdir(d)) <= 64 << 20
    for name, v in outputs.items():
        assert np.array_equal(np.load(os.path.join(d, name + ".npy")), v)
    with pytest.raises(AssertionError):
        bench.write_outputs(d, {"iter": np.array([3], np.int32)})
