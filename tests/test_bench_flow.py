"""bench.py's DataStream legs (Q3, Q5, as-of, Parquet) run end to end on the numpy kernel shim with the oracle
generator standing in for the CUDA generator: the Python of the benchmark -- program construction, timing loop,
result fields, flags -- is exercised in the CPU container; the numbers it prints here mean nothing."""
import os
import sys
import types

import numpy as np
import pytest
import torch

import cpu_shim
from oracle import tpch_gen as G

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def install(patch):
    """Routes bench.py onto the shim: `patch.setattr(obj, name, value)` (pytest's monkeypatch, or the plain setter the
    2-rank gloo worker of tests/test_dist_gloo.py uses).  Returns the bench module."""
    cpu_shim.install(patch)
    import quokka_b200.df as D
    import quokka_b200.runtime as RT
    from quokka_b200 import synth
    patch.setattr(D, "_default_device", lambda: torch.device("cpu"))
    patch.setattr(RT, "_default_device", lambda: torch.device("cpu"))
    patch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    patch.setattr(torch.cuda, "empty_cache", lambda *a, **k: None)
    gens = {"l_": ("lineitem", G.gen_lineitem), "o_": ("orders", G.gen_orders), "c_": ("customer", G.gen_customer), "s_": ("supplier", G.gen_supplier)}

    def column(name, sf, lo=0, hi=None, device=None):
        tab, fn = gens[name[:2]]
        hi = synth.sizes(sf)[tab] if hi is None else hi
        return torch.from_numpy(np.ascontiguousarray(fn(sf, lo, hi, [name])[name]))

    def ticks(table_id, n, n_symbols, lo=0, hi=None, gap=1000, columns=None, device=None):
        t = G.gen_ticks(table_id, n, n_symbols, lo, hi, gap)
        return {c: torch.from_numpy(np.ascontiguousarray(t[c])) for c in (columns or t)}
    patch.setattr(synth, "column", column)
    patch.setattr(synth, "ticks", ticks)
    import bench
    return bench


@pytest.fixture
def bench_on_shim(monkeypatch):
    return install(monkeypatch)


def run_multi_rank_legs(world, rank):
    """Called by the gloo worker after init_process_group: the Q3 (strong and weak), Q5 and as-of legs over `world` ranks."""
    import bench
    cpu = torch.device("cpu")
    q3 = bench.run_q3(_args(), torch, cpu, world, rank)
    q3w = bench.run_q3(_args(), torch, cpu, world, rank, weak=True)
    q3r = bench.run_q3(_args(no_replicate_builds=True), torch, cpu, world, rank)
    assert q3["top1"] == q3r["top1"] and q3["rows_per_s"] > 0 and q3w["rows_per_s"] > 0
    assert bench.run_q5(_args(), torch, cpu, world, rank)["rows_per_s"] > 0
    r = bench.run_asof(_args(), torch, cpu, world, rank)
    assert r["trades_out"] == 20_000 * world // 5


def _args(**kw):
    base = dict(q3_sf=0.02, q3_steps=1, replicate_builds=False, no_replicate_builds=False, steps=1, asof_quotes=20_000, parquet_sf=0.02, chunk_rows=40_000, q5_sf=0.02, only_parquet=True, no_parquet=False)
    base.update(kw)
    return types.SimpleNamespace(**base)


def test_q3_q5_legs(bench_on_shim):
    cpu = torch.device("cpu")
    for flag in (False, True):
        q3 = bench_on_shim.run_q3(_args(replicate_builds=flag), torch, cpu, 1, 0)
        assert q3["rows_per_s"] > 0 and q3["top1"]["revenue"] > 0 and len(q3["all_seconds"]) >= 1
        q5 = bench_on_shim.run_q5(_args(replicate_builds=flag), torch, cpu, 1, 0)
        assert q5["rows_per_s"] > 0


def test_asof_leg(bench_on_shim):
    r = bench_on_shim.run_asof(_args(), torch, torch.device("cpu"), 1, 0)
    assert r["trades_out"] == 20_000 // 5 and r["rows_per_s"] > 0


def test_parquet_leg(bench_on_shim):
    r = bench_on_shim.run_parquet(_args(), torch, torch.device("cpu"), 1, 0)
    for codec in ("none", "snappy", "zstd"):
        for mode in ("host", "device"):
            assert r[f"{mode}_{codec}"].get("agrees") is True, r[f"{mode}_{codec}"]
        assert r[f"file_bytes_{codec}"] > 0


def test_headline_line(bench_on_shim, monkeypatch, capsys, tmp_path):
    """The default (headline) arm: warm-up, timed loop with events, untimed extra steps for the clock sampler, parity
    check, JSON line with every contract key, the last timed step's Q1 state written by --dump-outputs.  CUDA events /
    devices are faked; the e2e leg (pinned memory) is off."""
    import json
    import quokka_b200

    class FakeEvent:
        def __init__(self, enable_timing=False): pass
        def record(self, stream=None): pass
        def elapsed_time(self, other): return 2.0

    monkeypatch.setattr(quokka_b200, "ops", cpu_shim, raising=False)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a, **k: None)
    real_device = torch.device
    monkeypatch.setattr(torch, "device", lambda *a, **k: real_device("cpu"))
    monkeypatch.setenv("WORLD_SIZE", "1")
    args = types.SimpleNamespace(sf=0.01, steps=3, warmup=3, variant=0, no_e2e=True, no_q3=False, no_cpu=False, extras=1, cpu_rows=200_000,
                                 only_q3=False, only_asof=False, only_q5=False, only_parquet=False, q3_sf=0.01, q3_steps=1, replicate_builds=False, no_replicate_builds=False,
                                 asof_quotes=10_000, e2e_rows=1000, e2e_chunk=1000, parquet_sf=0.01, chunk_rows=0, q5_sf=0.01, no_parquet=False,
                                 dump_outputs=str(tmp_path / "out"))
    bench_on_shim.run_ours(args)
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
                "data", "config", "roofline", "cpu_baseline", "e2e", "gpu_launches", "clocks", "parity", "q3", "q5", "asof"):
        assert key in line, key
    assert line["metric"] == "tpch_q1_rows_per_s" and line["n_gpus"] == 1 and line["steps"] == 3 and line["scaling"] == "weak"
    assert line["parity"]["ok"] is True and line["roofline"]["bound"] == "hbm" and line["cpu_baseline"]["kind"] == "port"
    assert "error" not in (line["q3"] or {}) and "error" not in (line["q5"] or {}) and "error" not in (line["asof"] or {})
    sums, counts = (np.load(str(tmp_path / "out" / f"{n}.npy")) for n in ("q1_sums", "q1_counts"))
    assert sums.dtype == counts.dtype == np.float64 and sums.shape == (6, 5) and counts.shape == (6,)
    assert int(counts.sum()) == line["parity"]["sum_of_group_counts"] == line["parity"]["rows_passing_filter"]
    li = G.gen_lineitem(0.01, columns=["l_shipdate", "l_quantity"])
    assert np.isclose(sums[:, 0].sum(), li["l_quantity"][li["l_shipdate"] <= G.DAY_1998_09_02].sum(), rtol=1e-12)
