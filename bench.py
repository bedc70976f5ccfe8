#!/usr/bin/env python
"""bench.py -- TPC-H Q1 (scan + filter + project + aggregate) throughput on synthetic TPC-H-shaped
lineitem, the metric BASELINE.json names: rows/s + achieved HBM GB/s, next to the CPU reference arm.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--sf 100]           (our arm)
  python bench.py --impl reference [...]                                     (CPU arm: Arrow/Acero)
  torchrun --nproc-per-node N bench.py --gpus N ...                          (one rank per GPU, NCCL)
  python bench.py [...] --dump-outputs DIR     (also writes the last timed step's Q1 result as DIR/*.npy)

A step = one pass of Q1 over this rank's lineitem shard.  Weak scaling: every rank holds its own
SF-`sf` shard (600 037 902 rows at SF-100, 22.8 GB of Q1 columns resident in HBM); the only data-path
collective is one all-reduce of the 6x5 partial-state matrix.  Inputs are 180x larger than L2, so no
explicit L2 flush is needed between steps.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

Q1_COLS = ["l_shipdate", "l_returnflag", "l_linestatus", "l_quantity", "l_extendedprice", "l_discount", "l_tax"]
Q1_BYTES_PER_ROW = 38          # date32 4 + 2 x 1-byte codes + 4 x fp64 (SURVEY.md section 8d)
Q1_PRED = "l_shipdate <= date '1998-12-01' - interval '90' day"
Q1_AGGS = ["l_quantity", "l_extendedprice", "l_extendedprice * (1 - l_discount)",
           "l_extendedprice * (1 - l_discount) * (1 + l_tax)", "l_discount"]
METRIC = "tpch_q1_rows_per_s"


def profiled_traffic_bytes():
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the committed
    `ncu --set full` capture (profiles/r01_q1_fused_tma.txt); None when the summary is not there."""
    import re
    p = os.path.join(ROOT, "profiles", "r01_q1_fused_tma.txt")
    try:
        m = re.search(r"DRAM traffic ([0-9.]+) GB", open(p).read())
        return float(m.group(1)) * 1e9 if m else None
    except OSError:
        return None


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int = 0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
def cpu_q1_arm(n_rows: int, steps: int, warmup: int, row_lo: int = 0):
    """Times the CPU restatement of the reference path (Arrow compute + Acero hash aggregate, all
    host threads) on a bounded sample of the same synthetic lineitem.  Returns (rows/s, info)."""
    import numpy as np
    import pyarrow as pa
    from concurrent.futures import ThreadPoolExecutor
    from oracle import queries as OQ
    from oracle import tpch_gen as G

    cores = os.cpu_count() or 1
    pa.set_cpu_count(cores)
    chunk = 2_000_000
    bounds = [(lo, min(lo + chunk, row_lo + n_rows)) for lo in range(row_lo, row_lo + n_rows, chunk)]
    with ThreadPoolExecutor(max_workers=min(cores, 32)) as ex:
        parts = list(ex.map(lambda b: G.gen_lineitem(100, b[0], b[1], Q1_COLS), bounds))
    cols = {c: np.concatenate([p[c] for p in parts]) for c in Q1_COLS}
    del parts
    tbl = G.to_arrow(cols)
    for _ in range(warmup):
        OQ.q1_acero_batched(tbl, threads=cores)
    passes = []
    for _ in range(steps):
        t0 = time.perf_counter()
        res = OQ.q1_acero_batched(tbl, threads=cores)
        passes.append(time.perf_counter() - t0)
    dt = min(passes)                 # best of k: the host arm is noisy (other tenants, NUMA placement); the best pass is the fairest
    info = {"kind": "port", "cores": cores, "unit": "rows/s",
            "sample": f"Q1 as the reference runs it on CPU (per-batch filter + projection + partial aggregate on a "
                      f"{cores}-thread pool, 2 M-row batches, then the final aggregate) with Arrow compute / Acero, on "
                      f"{n_rows} synthetic SF-100-shaped lineitem rows in RAM, {steps} timed passes",
            "groups": res.num_rows, "ms_per_pass": dt * 1e3, "all_ms": [round(x * 1e3, 1) for x in passes], "statistic": "best pass"}
    return n_rows / dt, info


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.cpu_rows
    v, info = cpu_q1_arm(n, max(1, args.steps), max(1, min(args.warmup, 2)))
    info["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": info["ms_per_pass"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "TPC-H Q1 scan+filter+aggregate, synthetic SF-100-shaped lineitem (bounded CPU sample)",
                       "rows_per_step": n, "bytes_per_row": Q1_BYTES_PER_ROW},
            "cpu_baseline": info,
            "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def dump_outputs(out_dir: str, arrays: dict):
    """Writes each tensor as out_dir/<name>.npy in float64 (the Q1 counts stay exact: they are far below 2^53), so that
    two builds can be compared output for output on the same seeded inputs."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().cpu().numpy().astype(np.float64))


def bind_to_gpu_numa_node(local: int):
    """Pin this rank's host threads to the CPUs of its GPU's NUMA node BEFORE any pinned buffer is allocated (first touch puts
    the pages there): at 8 ranks the end-to-end leg moves 8 x 55 GB/s out of host memory, and buffers on the wrong socket cross
    the inter-socket link (round 1: 538 ms per step at 8 GPUs against 413 ms at <= 4).  Best effort; returns what it did."""
    try:
        import pynvml
        pynvml.nvmlInit()
        bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(local)).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        bus = bus[-12:] if len(bus) > 12 else bus                     # 00000000:1b:00.0 -> 0000:1b:00.0
        node = int(open(f"/sys/bus/pci/devices/{bus}/numa_node").read().strip())
        if node < 0:
            return {"numa_node": None}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus |= set(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus)}
    except Exception as e:                                            # no NVML / sysfs entry: leave the affinity alone
        return {"numa_node": None, "why": f"{type(e).__name__}"}


# ---------------------------------------------------------------------------------------------
def run_ours(args):
    import torch
    import torch.distributed as dist
    from quokka_b200 import _lib as L, expr as E, ops, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # 3 channels x 6 GiB of mailbox per rank (of 180 GB): the 17 GB-per-rank as-of shuffle goes in 6 rounds instead of 18
        os.environ.setdefault("QK_MAILBOX_MB", "6144")
    numa = bind_to_gpu_numa_node(local) if world > 1 else {"numa_node": None, "why": "single rank: all host cores stay available"}
    if world > 1:
        import datetime
        # a rank-local failure must surface as an error within minutes, not as a silent hang of its peers
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=240))
    L.lib()

    if args.only_asof:
        r = run_asof(args, torch, dev, world, rank)
        if rank == 0:
            print(json.dumps({"asof": r}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.only_q5:
        r = run_q5(args, torch, dev, world, rank)
        if rank == 0:
            print(json.dumps({"q5": r}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.only_parquet:
        r = run_parquet(args, torch, dev, world, rank)
        if rank == 0:
            print(json.dumps({"parquet": r}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return
    if args.only_q3:
        q3 = run_q3(args, torch, dev, world, rank)
        if rank == 0:
            if q3.get("top1") and "o_orderdate" in q3["top1"]:
                q3["top1"]["o_orderdate"] = str(q3["top1"]["o_orderdate"])
            print(json.dumps({"q3": q3}), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    sf = args.sf
    n_total = synth.sizes(sf)["lineitem"]
    # weak scaling: each rank scans its own SF-`sf` shard, i.e. rows [rank*n_total, (rank+1)*n_total) of the
    # endless generator (same distribution, different rows)
    lo = rank * n_total
    cols = [synth.column(c, sf, lo, lo + n_total, device=dev) for c in Q1_COLS]
    torch.cuda.synchronize()

    sch = {c: E.ColumnInfo(i, ops.qk_dtype(t)) for i, (c, t) in enumerate(zip(Q1_COLS, cols))}
    pred = E.compile_expr(E.parse(Q1_PRED), sch)
    aggs = [E.compile_expr(E.parse(a), sch) for a in Q1_AGGS]
    gcols = [sch["l_returnflag"].slot, sch["l_linestatus"].slot]
    state = ops.DenseAggState([3, 2], [L.AGG_SUM] * 5, dev)

    def step():
        state.acc.zero_(); state.cnt.zero_()
        state.update(cols, pred, gcols, aggs, variant=args.variant)
        if world > 1:                                  # final merge of the 6x5 partial states
            dist.all_reduce(state.acc); dist.all_reduce(state.cnt)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step()
    barrier()
    variant_name = ops.last_variant() + "[" + ops.last_variant_config() + "]"
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    barrier()
    t_start.record()
    for i in range(args.steps):
        state.acc.zero_(); state.cnt.zero_()
        kev[i][0].record()
        state.update(cols, pred, gcols, aggs, variant=args.variant)
        kev[i][1].record()
        if world > 1:
            dist.all_reduce(state.acc); dist.all_reduce(state.cnt)
    t_end.record()
    barrier()
    if args.dump_outputs and rank == 0:                # the last timed step's result, before any untimed step touches it
        dump_outputs(args.dump_outputs, {"q1_sums": state.acc, "q1_counts": state.cnt})
    total_ms = t_start.elapsed_time(t_end)
    kern_ms = sum(a.elapsed_time(b) for a, b in kev) / args.steps
    launches = ops.launch_count() - launches0
    if world > 1:
        t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    # nvidia-smi samples every 100 ms: when the timed region is shorter than ~0.5 s keep the identical load running
    # (untimed) so that the clock / throttle record has a few samples taken under exactly this kernel.  The count
    # is derived from the max-over-ranks time, so every rank runs the same number of (collective) steps.
    extra_steps = 0
    if total_ms < 500.0:
        extra_steps = int((600.0 - total_ms) / max(total_ms / args.steps, 1e-3)) + 1
        for _ in range(extra_steps):
            step()
        barrier()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["sampled_over"] = f"the {args.steps} timed steps" + (f" + {extra_steps} identical untimed steps" if extra_steps else "")
    ms_per_step = total_ms / args.steps
    value = world * n_total / (ms_per_step / 1e3)

    # ---- result sanity at full size: every row is in exactly one group, counts add up to the filter count
    shipdate = cols[0]
    expect_rows = int((shipdate <= 10471).sum().item())
    got_rows = int(state.cnt.sum().item())             # after the all-reduce: rows of ALL ranks
    if world > 1:
        t = torch.tensor([expect_rows], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        expect_rows = int(t.item())
    parity_ok = got_rows == expect_rows
    # ... and the sums themselves: this rank's last step recomputed with torch in fp64 (a different summation order:
    # agreement within 1e-9 relative is the north_star tolerance), on a fresh single-rank state
    chk = ops.DenseAggState([3, 2], [L.AGG_SUM] * 5, dev)
    chk.update(cols, pred, gcols, aggs, variant=args.variant)
    sums_rel = 0.0
    mask = shipdate <= 10471
    gid = (cols[1].to(torch.int64) * 2 + cols[2].to(torch.int64))[mask]
    qty, price, disc, tax = (c[mask] for c in cols[3:7])
    for j, v in enumerate((qty, price, price * (1 - disc), price * (1 - disc) * (1 + tax), disc)):
        for g_ in range(6):          # one pairwise (tree) reduction per group: an accurate fp64 reference (atomic index_add_ is not)
            sel = gid == g_
            if not bool(sel.any()):
                continue
            ref = float(v[sel].sum(dtype=torch.float64).item())
            got = float(chk.acc[g_, j].item())
            if ref != 0.0:
                sums_rel = max(sums_rel, abs(got - ref) / abs(ref))
            del sel
        del v
    cnt_ok = bool((torch.bincount(gid, minlength=6) == chk.cnt).all().item())
    del mask, gid, qty, price, disc, tax, chk
    torch.cuda.empty_cache()
    parity_ok = parity_ok and cnt_ok and sums_rel <= 1e-9

    # ---- Q6's aggregate (three range terms, one on an fp64 column; sum(l_extendedprice * l_discount)) on the same resident columns:
    #      not one of the typed plans -> the runtime-described plan over the same TMA tile ring (fused_tma:dyn)
    q6 = None
    try:
        q6_pred = E.compile_expr(E.parse("l_shipdate >= date '1994-01-01' and l_shipdate < date '1995-01-01' and "
                                         "l_discount between 0.05 and 0.07 and l_quantity < 24"), sch)
        q6_agg = [E.compile_expr(E.parse("l_extendedprice * l_discount"), sch)]
        s6 = ops.DenseAggState([], [L.AGG_SUM], dev)
        for _ in range(3):
            s6.update(cols, q6_pred, [], q6_agg)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s6.acc.zero_(); s6.cnt.zero_()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            s6.update(cols, q6_pred, [], q6_agg)
        e1.record()
        torch.cuda.synchronize()
        ms6 = e0.elapsed_time(e1) / 10
        m6 = (cols[0] >= 8766) & (cols[0] < 9131) & (cols[5] >= 0.05) & (cols[5] <= 0.07) & (cols[3] < 24)
        ref6 = float((cols[4][m6] * cols[5][m6]).sum(dtype=torch.float64).item())
        got6 = float(s6.acc[0, 0].item()) / 10
        q6 = {"workload": "TPC-H Q6 partial aggregate on the resident SF-100 lineitem columns (4 columns, 28 B/row)", "kernel": ops.last_variant() + "[" + ops.last_variant_config() + "]",
              "ms": ms6, "rows_per_s": n_total / (ms6 / 1e3), "roofline": _roofline(n_total * 28, ms6 / 1e3, "28 B per lineitem row (date32 + 3 x fp64) over the kernel's time"),
              "rows_passing": int(s6.cnt[0].item()) // 10, "rows_passing_torch": int(m6.sum().item()),
              "rel_err_vs_torch_fp64": abs(got6 - ref6) / abs(ref6) if ref6 else 0.0}
        if args.dyn_sweep:                              # development: every tile shape of the dynamic plan, on Q6 and on Q1 forced through it
            sweep = {}
            for shape in ("256x4", "128x4", "256x2", "128x8", "128x2"):
                os.environ["QK_DYN_SHAPE"] = shape
                for name, st_, call in (("q6", s6, lambda: s6.update(cols, q6_pred, [], q6_agg)),
                                        ("q1", state, lambda: state.update(cols, pred, gcols, aggs, variant=7))):
                    for _ in range(2):
                        call()
                    torch.cuda.synchronize()
                    e0.record()
                    for _ in range(5):
                        call()
                    e1.record()
                    torch.cuda.synchronize()
                    sweep[f"{name}:{shape}"] = [round(e0.elapsed_time(e1) / 5, 3), ops.last_variant_config()]
            os.environ.pop("QK_DYN_SHAPE", None)
            q6["shape_sweep_ms"] = sweep
        del m6, s6
        torch.cuda.empty_cache()
    except Exception as e:                              # an extra must never take the headline line down
        q6 = {"error": f"{type(e).__name__}: {e}"[:300]}

    # ---- end to end through the operator API with HOST buffers (pinned), H2D inside the timed region
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, torch, dev, cols, world, rank)

    # ---- Q3 (shuffled joins) as an extra line item
    q3 = None
    if not args.no_q3:
        del cols
        torch.cuda.empty_cache()
        try:
            q3 = run_q3(args, torch, dev, world, rank)
            if q3 and q3.get("top1") and "o_orderdate" in q3["top1"]:
                q3["top1"]["o_orderdate"] = str(q3["top1"]["o_orderdate"])
            if world > 1:                               # SF-`q3_sf` PER GPU: the weak-scaling counterpart
                torch.cuda.empty_cache()
                q3w = run_q3(args, torch, dev, world, rank, weak=True)
                q3w["top1"]["o_orderdate"] = str(q3w["top1"]["o_orderdate"])
                q3["weak"] = q3w
        except Exception as e:                          # an extra must never take the headline line down
            q3 = {"error": f"{type(e).__name__}: {e}"[:300]}

    extras = {}
    if not args.no_q3 and args.extras >= 1:
        torch.cuda.empty_cache()
        legs = [("q5", run_q5), ("asof", run_asof)] + ([("e2e_parquet", run_parquet)] if (world == 1 and args.extras >= 1 and not args.no_parquet) else [])
        for name, fn in legs:
            try:
                extras[name] = fn(args, torch, dev, world, rank)
            except Exception as e:                      # extras must never take the headline line down
                extras[name] = {"error": f"{type(e).__name__}: {e}"[:300]}
            torch.cuda.empty_cache()

    # ---- CPU baseline (rank 0, N=1 only): bounded sample of the same workload
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        v, info = cpu_q1_arm(args.cpu_rows, 3, 1)
        info["value"] = v
        cpu = info

    if rank == 0:
        peak, peak_src = measured_peak_gbs()
        ach = n_total * Q1_BYTES_PER_ROW / (kern_ms / 1e3) / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"TPC-H Q1 SF-{sf:g} scan+filter+aggregate, {n_total} lineitem rows per GPU resident in HBM",
                       "rows_per_gpu": n_total, "bytes_per_row": Q1_BYTES_PER_ROW, "kernel": variant_name,
                       "l2": "inputs (22.8 GB) are larger than L2; no flush needed", "parallelism": f"shard x{world}, 1 all-reduce of 6x5 partials"},
            "gb_per_s": value * Q1_BYTES_PER_ROW / 1e9,
            "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                         "traffic": profiled_traffic_bytes() if (sf == 100 and "fused_tma:q1" in variant_name) else None,
                         "traffic_source": "profiles/r01_q1_fused_tma.txt (ncu --set full, same kernel and size)", "kernel": variant_name, "kernel_ms": kern_ms, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": n_total * Q1_BYTES_PER_ROW},
            "cpu_baseline": cpu, "e2e": e2e, "q6": q6, "q3": q3, "q5": extras.get("q5"), "asof": extras.get("asof"),
            "e2e_parquet": extras.get("e2e_parquet"),
            "gpu_launches": launches, "clocks": clocks, "host_binding": numa,
            "parity": {"rows_passing_filter": expect_rows, "sum_of_group_counts": got_rows,
                       "sums_vs_torch_fp64_max_rel_err": sums_rel, "group_counts_equal_torch_bincount": cnt_ok, "tolerance": 1e-9, "ok": parity_ok},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def run_q3(args, torch, dev, world, rank, weak=False):
    """TPC-H Q3 (lineitem x orders x customer hash joins + group-by + top-10) through the DataStream API on
    device-resident synthetic shards: SF-`q3_sf` in TOTAL, split evenly over the ranks (strong scaling); every
    join input and the partial aggregates are hash-partitioned and exchanged with NCCL all-to-all."""
    import torch.distributed as dist
    from quokka_b200 import synth
    from quokka_b200.columns import DeviceColumn, DeviceTable
    from quokka_b200.df import QuokkaContext
    import pyarrow as pa
    sf = args.q3_sf * (world if weak else 1)        # weak: SF-`q3_sf` per GPU
    sz = synth.sizes(sf)

    def shard(names, total):
        lo, hi = total * rank // world, total * (rank + 1) // world
        cols = {}
        for n in names:
            t = synth.column(n, sf, lo, hi, device=dev)
            cols[n] = DeviceColumn(t, synth.DICTIONARIES.get(n), pa.date32() if n in synth.DATE_COLUMNS else None)
        return DeviceTable(cols)

    li = shard(["l_orderkey", "l_shipdate", "l_extendedprice", "l_discount"], sz["lineitem"])
    od = shard(["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"], sz["orders"])
    cu = shard(["c_custkey", "c_mktsegment"], sz["customer"])
    torch.cuda.synchronize()

    def once():
        qc = QuokkaContext()
        qc.set_config("broadcast_cost_based", not args.no_replicate_builds)     # default: replicate a build side when that moves fewer rows
        br = args.chunk_rows or None
        lineitem, orders, customer = qc.from_device(li, batch_rows=br), qc.from_device(od, batch_rows=br), qc.from_device(cu, batch_rows=br)
        d = lineitem.join(orders, left_on="l_orderkey", right_on="o_orderkey")
        d = customer.join(d, left_on="c_custkey", right_on="o_custkey")
        d = d.filter_sql("c_mktsegment = 'BUILDING' and o_orderdate < date '1995-03-15' and l_shipdate > date '1995-03-15'")
        g = d.groupby(["l_orderkey", "o_orderdate", "o_shippriority"]).agg_sql("sum(l_extendedprice * (1 - l_discount)) as revenue")
        res = g.top_k(["revenue", "o_orderdate"], 10, descending=[True, False]).collect()
        return res, qc.last_graph

    import gc
    res, g = once()                       # warm-up (allocator, NCCL channels)
    if os.environ.get("QK_CPROFILE") and rank == 0:          # where does the HOST time of one query go?
        import cProfile, pstats, io
        once()
        pr = cProfile.Profile()
        pr.enable()
        once()
        torch.cuda.synchronize()
        pr.disable()
        buf = io.StringIO()
        pstats.Stats(pr, stream=buf).sort_stats("cumulative").print_stats(45)
        open(os.environ["QK_CPROFILE"], "w").write(buf.getvalue())
    elif os.environ.get("QK_CPROFILE"):
        once(); once()
    times = []
    for _ in range(max(1, args.q3_steps)):
        res = g = None
        gc.collect()                      # executor state of the previous run (hash tables, build sides) is garbage
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res, g = once()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        times.append(dt)
    dt = min(times)
    sent = torch.tensor([g.exchange.bytes_sent], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(sent)
    scan_bytes = sz["lineitem"] * 28 + sz["orders"] * 24 + sz["customer"] * 9
    return {"workload": f"TPC-H Q3 SF-{sf:g} total, {'weak' if weak else 'strong'} scaling over {world} GPU(s), DataStream API on HBM-resident shards",
            "rows_per_s": sz["lineitem"] / dt, "seconds": dt, "all_seconds": times, "lineitem_rows": sz["lineitem"],
            "scan_gb_per_s": scan_bytes / dt / 1e9, "scan_bytes": scan_bytes,
            "roofline": _roofline(scan_bytes / max(world, 1), dt, "Q3 scan bytes per GPU (28 B/lineitem row + 24 B/orders row + 9 B/customer row, SURVEY 8d) over the WHOLE query's wall time"),
            "shuffle_bytes_over_nvlink": float(sent.item()), "shuffle_gb_per_s_per_gpu": float(sent.item()) / max(world, 1) / dt / 1e9,
            "shuffle_frac_of_nvlink_900": float(sent.item()) / max(world, 1) / dt / 1e9 / 900.0,
            "exchanges": g.exchange.calls, "exchanges_via_peer_memory": g.exchange.peer_calls, "lanes": g.lanes_used, "chunk_rows": args.chunk_rows,
            "profile_ms": g.report() if g.profile else None,
            "top1": {k: (res[k][0].as_py() if res.num_rows else None) for k in res.column_names} if res is not None else None}


_LAST = {"qc": None}


def _last_graph_report():
    g = _LAST["qc"].last_graph if _LAST["qc"] is not None else None
    return g.report() if g is not None else None


def _roofline(bytes_per_gpu, seconds, what):
    peak, src = measured_peak_gbs()
    ach = bytes_per_gpu / seconds / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "algorithmic_bytes_per_gpu": bytes_per_gpu,
            "peak_source": src, "what": what}


def _timed_collect(torch, dist, dev, world, fn, steps):
    import gc
    fn()
    times = []
    for _ in range(max(1, steps)):
        gc.collect()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = fn()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([dt], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        times.append(dt)
    return res, min(times), times


def run_q5(args, torch, dev, world, rank):
    """TPC-H Q5 (apps/tpc-h/tpch.py:223-236): broadcast join with the 5 ASIA nations, three shuffled joins
    (orders, lineitem, supplier), post-join s_nationkey = c_nationkey, sum(revenue) by nation."""
    import pyarrow as pa
    import torch.distributed as dist
    from quokka_b200 import synth
    from quokka_b200.columns import DeviceColumn, DeviceTable
    from quokka_b200.df import QuokkaContext
    sf = args.q5_sf
    sz = synth.sizes(sf)

    def shard(names, total):
        lo, hi = total * rank // world, total * (rank + 1) // world
        return DeviceTable({n: DeviceColumn(synth.column(n, sf, lo, hi, device=dev), synth.DICTIONARIES.get(n),
                                            pa.date32() if n in synth.DATE_COLUMNS else None) for n in names})
    li = shard(["l_orderkey", "l_suppkey", "l_extendedprice", "l_discount"], sz["lineitem"])
    od = shard(["o_orderkey", "o_custkey", "o_orderdate"], sz["orders"])
    cu = shard(["c_custkey", "c_nationkey"], sz["customer"])
    su = shard(["s_suppkey", "s_nationkey"], sz["supplier"])
    na, re = synth.nation_table(), synth.region_table()

    def once():
        qc = QuokkaContext()
        qc.set_config("broadcast_cost_based", not args.no_replicate_builds)
        br = args.chunk_rows or None
        lineitem, orders, customer, supplier = (qc.from_device(t_, batch_rows=br) for t_ in (li, od, cu, su))
        nation, region = qc.from_arrow(na), qc.from_arrow(re)
        asia = region.filter_sql("r_name == 'ASIA'")
        asian = nation.join(asia, left_on="n_regionkey", right_on="r_regionkey").select(["n_name", "n_nationkey"])
        d = customer.join(asian, left_on="c_nationkey", right_on="n_nationkey")
        d = d.join(orders, left_on="c_custkey", right_on="o_custkey", suffix="_3")
        d = d.join(lineitem, left_on="o_orderkey", right_on="l_orderkey", suffix="_4")
        d = d.join(supplier, left_on="l_suppkey", right_on="s_suppkey", suffix="_5")
        d = d.filter_sql("s_nationkey = c_nationkey and o_orderdate >= date '1994-01-01' and o_orderdate < date '1994-01-01' + interval '1' year")
        return d.groupby("n_name").agg_sql("sum(l_extendedprice * (1 - l_discount)) as revenue").collect()

    res, dt, times = _timed_collect(torch, dist, dev, world, once, args.q3_steps)
    rows = sorted(zip(res["n_name"].to_pylist(), res["revenue"].to_pylist()), key=lambda x: -x[1])
    scan_bytes = sz["lineitem"] * 32 + sz["orders"] * 20 + sz["customer"] * 16 + sz["supplier"] * 16
    return {"workload": f"TPC-H Q5 SF-{sf:g} total (strong scaling) over {world} GPU(s), DataStream API on HBM-resident shards",
            "rows_per_s": sz["lineitem"] / dt, "seconds": dt, "all_seconds": times, "result": rows, "lineitem_rows": sz["lineitem"],
            "scan_bytes": scan_bytes, "scan_gb_per_s": scan_bytes / dt / 1e9,
            "roofline": _roofline(scan_bytes / max(world, 1), dt, "Q5 scan bytes per GPU (32 B/lineitem + 20 B/orders + 16 B/customer + 16 B/supplier row, SURVEY 8d) over the whole query's wall time"),
            "chunk_rows": args.chunk_rows}


def run_asof(args, torch, dev, world, rank):
    """trades.join_asof(quotes, on=time, by=symbol) -> sum(cast(asize*100 as int)) (apps/tpc-h/range.py:10-16) on
    SIP-shaped synthetic ticks generated in HBM: each rank holds a contiguous time range of both streams."""
    import torch.distributed as dist
    from quokka_b200 import synth
    from quokka_b200.columns import DeviceColumn, DeviceTable
    from quokka_b200.df import QuokkaContext
    nq, nt, nsym = args.asof_quotes * world, args.asof_quotes * world // 5, 8000
    qlo, qhi = nq * rank // world, nq * (rank + 1) // world
    tlo, thi = nt * rank // world, nt * (rank + 1) // world
    # same time axis for both streams: 5 quotes per trade on average
    quotes = DeviceTable({k: DeviceColumn(v) for k, v in synth.ticks(synth.T_QUOTES, nq, nsym, qlo, qhi, gap=1000, columns=["time", "symbol", "asize"], device=dev).items()})
    trades = DeviceTable({k: DeviceColumn(v) for k, v in synth.ticks(synth.T_TRADES, nt, nsym, tlo, thi, gap=5000, columns=["time", "symbol", "size"], device=dev).items()})

    def once():
        qc = QuokkaContext()
        _LAST["qc"] = qc
        t = qc.from_device(trades, sorted_by="time")
        q = qc.from_device(quotes, sorted_by="time")
        return t.join_asof(q, on="time", by="symbol").agg_sql("sum(cast(asize * 100 as int)) as s, count(*) as n").collect()

    res, dt, times = _timed_collect(torch, dist, dev, world, once, 2)
    if os.environ.get("QK_PROFILE") and rank == 0:
        from quokka_b200.df import QuokkaContext as _QC
        print("asof profile_ms:", json.dumps(_last_graph_report()), file=sys.stderr, flush=True)
    alg = 12 * (nq + nt) + 8 * nt                 # time 8 B + by-code 4 B per row of both sides; per trade: gathered asize 4 B + 4 B written
    # the join kernels alone (qk_asof_merge: bounds + local + carry + sweep) on this rank's resident columns, CUDA events
    kernel = None
    try:
        from quokka_b200 import ops
        lt, lb = trades["time"].data, trades["symbol"].data.to(torch.int32)
        rt, rb = quotes["time"].data, quotes["symbol"].data.to(torch.int32)
        for _ in range(2):
            ops.asof_merge(lt, lb, rt, rb, nsym)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            ridx, _c = ops.asof_merge(lt, lb, rt, rb, nsym)
        e1.record()
        torch.cuda.synchronize()
        kms = e0.elapsed_time(e1) / 5
        kalg = 12 * (rt.numel() + lt.numel()) + 4 * lt.numel()           # both sides read once (time + key), 4 B written per left row
        kernel = {"ms": kms, "rows_per_s": (rt.numel() + lt.numel()) / (kms / 1e3), "matched": int((ridx >= 0).sum().item()),
                  "roofline": _roofline(kalg, kms / 1e3, "qk_asof_merge alone: 12 B per row of both sides + 4 B per left row over the four kernels' time")}
        del ridx, lb, rb
    except Exception as e:
        kernel = {"error": f"{type(e).__name__}: {e}"[:300]}
    return {"workload": f"as-of join, {nt} trades x {nq} quotes in total ({(nq + nt) / 1e9:.2f} B rows), {nsym} symbols, {world} GPU(s), weak scaling "
                        f"({args.asof_quotes} quotes per GPU, each rank a contiguous time range)", "rows_per_s": (nq + nt) / dt,
            "seconds": dt, "all_seconds": times, "checksum": res["s"][0].as_py(), "trades_out": res["n"][0].as_py(),
            "roofline": _roofline(alg / max(world, 1), dt, "12 B per row of both sides + 8 B per trade (SURVEY 8d) over the whole DataStream program's wall time"),
            "join_kernels": kernel}


def run_e2e(args, torch, dev, cols, world, rank):
    """Same metric through the PUBLIC API with HOST buffers: pinned Arrow-layout columns ->
    QuokkaContext.from_pinned(...).filter_sql(...).groupby(...).agg_sql(...).collect().  Every step copies the
    step's inputs host->device (chunked, double-buffered against the fused kernel) and brings the result back
    as a pyarrow.Table."""
    import torch.distributed as dist
    from quokka_b200 import synth
    from quokka_b200.df import QuokkaContext
    n = min(cols[0].numel(), args.e2e_rows)
    host = {}
    for name, t in zip(Q1_COLS, cols):
        h = torch.empty(n, dtype=t.dtype, pin_memory=True)
        h.copy_(t[:n])
        host[name] = h
    torch.cuda.synchronize()
    dicts = {c: synth.DICTIONARIES[c] for c in ("l_returnflag", "l_linestatus")}
    sql = ("sum(l_quantity) as sum_qty, sum(l_extendedprice) as sum_base_price, sum(l_extendedprice * (1 - l_discount)) as sum_disc_price, "
           "sum(l_extendedprice * (1 - l_discount) * (1 + l_tax)) as sum_charge, avg(l_quantity) as avg_qty, "
           "avg(l_extendedprice) as avg_price, avg(l_discount) as avg_disc, count(*) as count_order")

    def once():
        qc = QuokkaContext()
        qc.set_config("pinned_chunk_rows", args.e2e_chunk)
        s = qc.from_pinned(host, dictionaries=dicts, dates=("l_shipdate",))
        return s.filter_sql(Q1_PRED).groupby(["l_returnflag", "l_linestatus"]).agg_sql(sql).collect()

    res, dt, times = _timed_collect(torch, dist, dev, world, once, max(1, min(args.steps, 5)))
    rows = int(sum(res["count_order"].to_pylist()))
    d2h = sum(c.nbytes for c in res.columns)
    return {"value": world * n / dt, "unit": "rows/s", "h2d_bytes_per_step": n * Q1_BYTES_PER_ROW,
            "d2h_bytes_per_step": int(d2h), "rows_per_step_per_gpu": n, "ms_per_step": dt * 1e3, "all_ms": [t * 1e3 for t in times],
            "result_rows": res.num_rows, "count_order_total": rows,
            "note": "QuokkaContext.from_pinned(...).filter_sql().groupby().agg_sql().collect(): pinned host Arrow-layout "
                    "columns -> chunked H2D on 2 copy streams, overlapped with the fused Q1 kernel -> final aggregate -> pyarrow.Table"}


def run_parquet(args, torch, dev, world, rank):
    """Q1 end to end FROM PARQUET FILES through `QuokkaContext.read_parquet` (not part of the default line):
    the reference's layout (row groups of 100 000, apps/convert.py:5-19), written here from the synthetic generator,
    read (a) with Arrow on the host + upload of decoded columns, as the reference's reader does, (b) with the pages
    decoded on the device (config device_parquet), for uncompressed and Snappy files.  Page cache warm."""
    import shutil
    import tempfile
    import pyarrow as pa
    import pyarrow.parquet as pq
    import torch.distributed as dist
    from quokka_b200 import synth
    from quokka_b200.df import QuokkaContext
    sf = args.parquet_sf
    n = synth.sizes(sf)["lineitem"]
    lo = rank * n
    root = tempfile.mkdtemp(prefix=f"qk_parquet_r{rank}_")
    out = {"sf_per_gpu": sf, "rows_per_gpu": n, "row_group_size": 100_000,
           "what": "Q1 END TO END FROM PARQUET FILES through QuokkaContext.read_parquet(...).filter_sql().groupby().agg_sql().collect(): file "
                   "bytes -> result, page cache warm; `host_*` = Arrow decodes on the host like the reference's reader "
                   "(unordered_readers.py:51,98-99), `device_*` = the encoded column chunks cross PCIe and are decoded in HBM (qk_parquet_*)"}
    try:
        arrays = {}
        for c in Q1_COLS:
            h = synth.column(c, sf, lo, lo + n, device=dev).cpu().numpy()
            if c in synth.DICTIONARIES:
                arrays[c] = pa.DictionaryArray.from_arrays(pa.array(h.astype("int8")), pa.array(synth.DICTIONARIES[c])).cast(pa.string())
            elif c in synth.DATE_COLUMNS:
                arrays[c] = pa.array(h, pa.int32()).cast(pa.date32())
            else:
                arrays[c] = pa.array(h)
        tbl = pa.table(arrays)
        sql = ("sum(l_quantity) as sum_qty, sum(l_extendedprice * (1 - l_discount)) as sum_disc_price, "
               "sum(l_extendedprice * (1 - l_discount) * (1 + l_tax)) as sum_charge, avg(l_discount) as avg_disc, count(*) as count_order")
        expect = None
        for codec in (("none", "snappy", "zstd") if args.only_parquet else ("none", "snappy")):
            path = os.path.join(root, f"lineitem_{codec}.parquet")
            pq.write_table(tbl, path, compression=None if codec == "none" else codec, row_group_size=100_000)
            out[f"file_bytes_{codec}"] = os.path.getsize(path)
            for mode in ("host", "device"):
                def once():
                    qc = QuokkaContext()
                    qc.set_config("device_parquet", mode == "device")
                    return qc.read_parquet(path).filter_sql(Q1_PRED).groupby(["l_returnflag", "l_linestatus"]).agg_sql(sql).collect()
                try:
                    res, dt, times = _timed_collect(torch, dist, dev, world, once, 3)
                    cnt = int(sum(res["count_order"].to_pylist()))
                    expect = cnt if expect is None else expect
                    out[f"{mode}_{codec}"] = {"rows_per_s": world * n / dt, "ms": dt * 1e3, "all_ms": [t * 1e3 for t in times],
                                              "count_order_total": cnt, "agrees": cnt == expect,
                                              "encoded_gb_per_s": out[f"file_bytes_{codec}"] / dt / 1e9, "decoded_gb_per_s": n * Q1_BYTES_PER_ROW / dt / 1e9}
                except Exception as e:
                    out[f"{mode}_{codec}"] = {"error": f"{type(e).__name__}: {e}"[:300]}
        del tbl, arrays
    finally:
        shutil.rmtree(root, ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--sf", type=float, default=100)
    ap.add_argument("--variant", type=int, default=0, help="0 auto, 1 generic, 2 fused LDG, 3 fused TMA")
    ap.add_argument("--cpu-rows", type=int, default=120_000_000)
    ap.add_argument("--e2e-rows", type=int, default=600_037_902)
    ap.add_argument("--e2e-chunk", type=int, default=16 * 1024 * 1024)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-q3", action="store_true")
    ap.add_argument("--dyn-sweep", action="store_true", help="development: time every tile shape of the dynamic fused plan")
    ap.add_argument("--only-q3", action="store_true")
    ap.add_argument("--only-asof", action="store_true")
    ap.add_argument("--only-q5", action="store_true")
    ap.add_argument("--only-parquet", action="store_true", help="time Q1 from Parquet files: host (Arrow) reader vs device decode")
    ap.add_argument("--parquet-sf", type=float, default=5)
    ap.add_argument("--replicate-builds", action="store_true", help="(default behaviour; kept for older command lines)")
    ap.add_argument("--no-replicate-builds", action="store_true",
                    help="Q3 / Q5: shuffle both sides of every join instead of replicating a build side when that moves fewer rows")
    ap.add_argument("--extras", type=int, default=1,
                    help="1: also time Q5 and the as-of join when running on one GPU; 2: at any GPU count; 0: never")
    ap.add_argument("--asof-quotes", type=int, default=1_050_000_000,
                    help="quote rows per GPU in the as-of extra (+ a fifth as many trades): 8 GPUs x 1.26 B = 10 B rows, BASELINE config 5")
    ap.add_argument("--q5-sf", type=float, default=300, help="scale factor of the Q5 extra (BASELINE config 4: SF-300), strong scaling")
    ap.add_argument("--no-parquet", action="store_true", help="skip the Parquet end-to-end leg of the default line (1 GPU only)")
    ap.add_argument("--q3-sf", type=float, default=100)
    ap.add_argument("--q3-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the Q1 state of the last timed step as DIR/q1_sums.npy (6 groups x 5 sums, "
                         "group = returnflag * 2 + linestatus) and DIR/q1_counts.npy, both float64 (rank 0)")
    ap.add_argument("--chunk-rows", type=int, default=0,
                    help="Q3 / Q5 readers emit chunks of this many rows (0 = one batch per shard); chunks are pipelined over lanes")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
