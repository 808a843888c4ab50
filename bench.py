#!/usr/bin/env python3
"""bench.py — headline benchmark of the B200-native roaring executor (contract: DESIGN.md §6).

Workload (BASELINE.json configs[1]): per GPU 1024 shards x 2^20 columns, 64 rows at 1 % density, one step =
    Count(Intersect(Union(Row(f=0..31)), Union(Row(f=32..63))))   over the GPU's whole shard batch
= 63 Row-level set-ops + 1 Count row per shard.  metric = set-ops/s (whole job, all GPUs); extras: Count rows/s,
columns/s, HBM GB/s vs the measured roofline.  The same JSON line carries sub-records for the other BASELINE configs,
each with its own roofline fraction, CPU baseline and parity check against the CPU port:
    north_star   configs[4] at the acceptance point: Count(Intersect(Row, Row)) at 1 %, 1 B columns per GPU — one query per
                 launch (rotating over 32 row pairs = 1.4 GB) and 32 pairs fused in one launch
    density_sweep  configs[4] around it: 0.01 % .. 50 % uniform and two clustered (run-container) points, same two forms, on every rank
    config3      BSI Count(Row(v > 2^31)) over 10 M records (rank 0)
    config4      GroupBy(Rows(a), Rows(b)) 256 x 256, 512 shards per GPU, ncclAllReduce of the 512 KiB count tensor at N > 1

  python bench.py --gpus 1 --steps 20 --warmup 3            # our arm (CUDA kernels through the C ABI)
  python bench.py --impl reference --steps 3 --warmup 1     # reference arm: CPU restatement on all host cores
  torchrun ... bench.py --gpus N ...                        # one rank per GPU, shards range-partitioned, merged count
  python bench.py --steps 20 --dump-outputs DIR             # also DIR/<name>.npy: what each timed query returned in its last step

The inputs are generated from fixed seeds, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the tree may be read-only where the benchmark runs: leave no __pycache__ in it

# name -> what a timed query returned to its caller in its last timed step (merged over ranks); --dump-outputs writes them
LAST_OUTPUTS = {}

FIELD_SEED_ID = 1
ROWS_A, ROWS_B = list(range(32)), list(range(32, 64))
SET_OPS_PER_SHARD = (len(ROWS_A) - 1) + (len(ROWS_B) - 1) + 1     # 31 + 31 unions, 1 intersect
SW = 1 << 20
WORKLOAD = "configs[1]: 1024 shards x 2^20 cols per GPU, 1% density, 64-row Union->Intersect->Count"
QUERY = "Count(Intersect(Union(Row f=0..31),Union(Row f=32..63)))"
PAIRS_A, PAIRS_B = list(range(0, 64, 2)), list(range(1, 64, 2))   # north-star row pairs (2k, 2k+1) of the same field


def query_text():
    ua = "Union(" + ", ".join(f"Row(f={r})" for r in ROWS_A) + ")"
    ub = "Union(" + ", ".join(f"Row(f={r})" for r in ROWS_B) + ")"
    return f"Count(Intersect({ua}, {ub}))"


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def build_cpu_side():
    """the pieces the CPU reference arm needs (datagen helper + oracle) — never the CUDA library"""
    from featurebase_b200 import build as B
    B.build_datagen()
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "libfboracle.so"], stdout=subprocess.DEVNULL)


class ClockSampler:
    """samples nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)"""

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc, self.t = gpu, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", "--query-gpu=clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.t = threading.Thread(target=self._read, daemon=True)
        self.t.start()

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------- CPU port (oracle/fb_bench.c)
class CpuArm:
    """the reference's algorithms on the host cores: long-lived pinned worker pool, rows handed out as views (no copies)"""

    def __init__(self):
        from oracle import oracle as O
        self.O = O
        self.threads = len(os.sched_getaffinity(0)) or os.cpu_count() or 1
        self.pool = O.Pool(self.threads, pin=True)
        self.calibration = None
        self.note = ("C restatement of the reference's roaring / executor algorithms (Go toolchain absent): persistent pool of %d threads, shards pulled "
                     "dynamically, fragment.row as views over frozen containers, no allocation of row payloads" % self.threads)

    def calibrate(self, frags, shards):
        """How many cores does this box really give the process?  One thread over 16 shards vs the whole pool over all of them, pinned and
        unpinned; the faster pool is kept.  (Round 1 saw the same binary at 100 ms and 25 ms per step on two leases of the same pool: a box
        that advertises 128 CPUs through a cgroup quota is not a 128-core host — parallel_speedup makes that visible.)"""
        O = self.O
        one = O.Pool(1, pin=False)
        n1 = min(16, len(frags))
        t1 = min(O.bench_union_intersect_count(one, frags[:n1], shards[:n1], ROWS_A, ROWS_B)[1] for _ in range(2)) / n1
        one.close()
        res = {}
        for pin in (True, False):
            pool = self.pool if pin else O.Pool(self.threads, pin=False)
            res[pin] = (min(O.bench_union_intersect_count(pool, frags, shards, ROWS_A, ROWS_B)[1] for _ in range(2)), pool)
        best = min(res, key=lambda k: res[k][0])
        for pin, (_, pool) in res.items():
            if pin != best:
                pool.close()
        self.pool = res[best][1]
        self.calibration = {"single_thread_ms_per_shard": t1 * 1e3, "threads": self.threads, "pinned": bool(best),
                            "parallel_speedup": t1 * len(frags) / res[best][0], "pinned_ms": res[True][0] * 1e3, "unpinned_ms": res[False][0] * 1e3}
        return self.calibration

    def fragments(self, bulk, n):
        return [self.O.Bitmap.from_bytes(bulk.fragment_bytes(i)) for i in range(n)]

    def headline(self, frags, shards, reps):
        times, count = [], None
        for _ in range(reps):
            count, secs = self.O.bench_union_intersect_count(self.pool, frags, shards, ROWS_A, ROWS_B)
            times.append(secs)
        return count, times

    def pairs(self, frags, shards, reps, materialise=True, rows_a=None, rows_b=None):
        times, counts = [], None
        for _ in range(reps):
            counts, secs = self.O.bench_pair_counts(self.pool, frags, shards, rows_a or PAIRS_A, rows_b or PAIRS_B, materialise)
            times.append(secs)
        return counts, times


def config_record(S, world, payload, reduce):
    """`config` of the JSON line — the same dict from both arms (the driver compares them)"""
    l2 = (f"inputs {payload / 1e6:.0f} MB per GPU > 126 MB L2 (no flush needed)" if payload > 126e6 else
          f"inputs {payload / 1e6:.0f} MB per GPU fit the 126 MB L2: NOT a valid bench size (use the default --shards-per-gpu)")
    return {"workload": WORKLOAD, "query": QUERY, "shards_per_gpu": S, "total_shards": S * world, "density": 0.01, "l2": l2,
            "parallelism": f"shard-range x{world}", "count_merge": (reduce if world > 1 else "none")}


def gen_headline(shards):
    from featurebase_b200 import datagen as D
    return D.fragments(FIELD_SEED_ID, shards, ROWS_A + ROWS_B, 0.01)


def run_reference(args):
    """bench.py --impl reference: the same workload on the host cores only (no CUDA library is loaded by this arm)"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    build_cpu_side()
    cpu = CpuArm()
    S = args.shards_per_gpu
    shards = np.arange(S, dtype=np.uint64)
    bulk = gen_headline(shards)
    frags = cpu.fragments(bulk, S)
    cpu.calibrate(frags, shards)
    # payload bytes of the 64 rows, from the fragments' own container tables (the GPU arm asks the library for the same figure)
    payload = 0
    for i in range(S):
        raw = bulk.buf[int(bulk.offsets[i]):int(bulk.offsets[i + 1])]
        n = int(np.frombuffer(raw[4:8], dtype="<u4")[0])
        hdr = np.frombuffer(raw[8:8 + 12 * n], dtype=np.dtype([("key", "<u8"), ("typ", "<u2"), ("n1", "<u2")]))
        arr = hdr["typ"] == 1
        payload += int(2 * (hdr["n1"][arr].astype(np.int64) + 1).sum()) + 8192 * int((hdr["typ"] == 2).sum())
        for j in np.nonzero(hdr["typ"] == 3)[0]:
            off = int(np.frombuffer(raw[8 + 12 * n + 4 * j: 12 + 12 * n + 4 * j], dtype="<u4")[0])
            payload += 4 * int(np.frombuffer(raw[off:off + 2], dtype="<u2")[0])
    if args.warmup:
        cpu.headline(frags, shards, min(args.warmup, 2))
    count, times = cpu.headline(frags, shards, max(args.steps, 1))
    sec = float(np.median(times))
    val = SET_OPS_PER_SHARD * S / sec
    pc, ptimes = cpu.pairs(frags, shards, 3)
    psec = float(np.median(ptimes))
    line = {
        "impl": "reference", "metric": "set_ops_per_sec", "value": val, "unit": "set-ops/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u64/u16 integer", "data": "synthetic",
        "config": config_record(S, max(args.gpus, 1), payload, args.reduce),
        "count_rows_per_sec": S / sec, "columns_per_sec": S * SW / sec,
        "cpu_baseline": {"value": val, "unit": "set-ops/s", "cores": cpu.threads, "kind": "port", "calibration": cpu.calibration,
                         "sample": f"{S} of the {S * max(args.gpus, 1)} shards (one GPU's share; throughput does not depend on the shard count), {len(times)} steps, median; " + cpu.note},
        "e2e": {"value": val, "unit": "set-ops/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "north_star": {"query": "32 x Count(Intersect(Row(f=2k), Row(f=2k+1))) over the same shards (executor path: Intersect materialises, Count sums)",
                       "ms": psec * 1e3, "set_ops_per_sec": len(PAIRS_A) * S / psec},
        "check_count": count,
    }
    if args.dump_outputs:
        LAST_OUTPUTS["headline_count"] = np.array([count], dtype=np.uint64)
        dump_outputs(args.dump_outputs)
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------- our arm
def timed_calls(ctx, fn, steps, warmup):
    for i in range(warmup):
        fn(i)
    ms = []
    t0 = time.perf_counter()
    for i in range(steps):
        fn(warmup + i)
        ms.append(ctx.counters()["last_query_gpu_ms"])
    wall = (time.perf_counter() - t0) / steps * 1e3
    return float(np.mean(ms)), float(np.min(ms)), wall


def pair_record(h, idx, fld, shards, rows_a, rows_b, label, name, cpu, frags, peak, world, dist, torch, steps):
    """Count(Intersect(Row a_k, Row b_k)) over this rank's shards: (i) one query per launch, rotating over the row pairs, (ii) all pairs
    fused in one launch (SURVEY §8d).  Parity of every pair's count against the CPU port over ALL shards (all ranks)."""
    from featurebase_b200 import executor as X, lib as L
    ctx = h.ctx
    progs = [[L.Op(L.OP_ROW, fld.id, 0, 0, a, 0, 0, 0), L.Op(L.OP_ROW, fld.id, 0, 0, b, 0, 0, 0), L.Op(L.OP_INTERSECT, 0, 0, 2, 0, 0, 0, 0)] for a, b in zip(rows_a, rows_b)]
    progs = [L.ops_array(p) for p in progs]
    n_pairs = len(progs)
    single = {}

    def one(i):
        single[i % n_pairs] = ctx.count(idx.id, progs[i % n_pairs], shards)

    n_single = max(4 * n_pairs, steps)
    if world > 1:
        # the ranks generate and load their own shards before this point (CPU work whose duration differs per rank, more so with N ranks
        # sharing the host cores); the fused Count merge waits for a peer inside the kernel for a bounded time only, so the ranks are
        # lined up before the first collective query
        dist.barrier()
    s_ms, s_min, s_wall = timed_calls(ctx, one, n_single, n_pairs)
    batched = {}

    def fused(i):
        batched[0] = ctx.count_pairs(idx.id, fld.id, 0, rows_a, fld.id, 0, rows_b, shards)

    b_ms, b_min, b_wall = timed_calls(ctx, fused, max(steps, 10), 3)
    pay, nc = ctx.rows_payload_bytes(idx.id, fld.id, X.VIEW_STANDARD, shards, list(rows_a) + list(rows_b))
    algo_all = pay + 16 * nc + 8 * n_pairs
    algo_one = algo_all / n_pairs
    got = np.asarray(batched[0], dtype=np.uint64)
    got_single = np.array([single[k] for k in range(n_pairs)], dtype=np.uint64)
    LAST_OUTPUTS[name + "_single"], LAST_OUTPUTS[name + "_batched"] = got_single, got
    names = ("absent", "array", "bitmap", "run")      # device-side analogue of the reference's statsHit("intersectionCount/...") counters
    hm = ctx.pair_types(idx.id, fld.id, 0, rows_a[0], fld.id, 0, rows_b[0], shards)
    hist = {"%s x %s" % (names[i], names[j]): int(hm[i][j]) for i in range(4) for j in range(4) if hm[i][j]}
    l2 = "%.2f GB touched per cycle (> L2)" % (algo_all / 1e9) if algo_all > 126e6 else "%.0f MB touched per cycle: fits the 126 MB L2 — a launch / L2-bound point, not an HBM one" % (algo_all / 1e6)
    rec = {"query": "Count(Intersect(Row(f=a), Row(f=b))), %s, %d shards x 2^20 columns per GPU" % (label, len(shards)),
           "single": {"ms": s_ms, "ms_min": s_min, "e2e_ms": s_wall, "gbs": algo_one / (s_ms * 1e-3) / 1e9, "frac": algo_one / (s_ms * 1e-3) / 1e9 / peak,
                      "algorithmic_bytes": int(algo_one), "launches_timed": n_single,
                      "note": "one fused pair_count_kernel launch per query, CUDA events around each launch; the %d row pairs are rotated: %s" % (n_pairs, l2)},
           "batched": {"ms": b_ms, "ms_min": b_min, "e2e_ms": b_wall, "pairs_per_launch": n_pairs, "gbs": algo_all / (b_ms * 1e-3) / 1e9, "frac": algo_all / (b_ms * 1e-3) / 1e9 / peak,
                       "algorithmic_bytes": int(algo_all), "note": "fbgpu_count_pairs: %d independent row pairs in one launch" % n_pairs},
           "set_ops_per_sec_single": len(shards) * world / (s_ms * 1e-3), "set_ops_per_sec_batched": n_pairs * len(shards) * world / (b_ms * 1e-3),
           "container_pair_types_pair0": hist}
    if world > 1:
        t = torch.tensor([s_ms, b_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)                  # max over ranks, like the headline
        for key, v in (("single", float(t[0])), ("batched", float(t[1]))):
            by = algo_one if key == "single" else algo_all
            rec[key].update({"ms": v, "gbs": by / (v * 1e-3) / 1e9, "frac": by / (v * 1e-3) / 1e9 / peak})
        rec["set_ops_per_sec_single"] = len(shards) * world / (float(t[0]) * 1e-3)
        rec["set_ops_per_sec_batched"] = n_pairs * len(shards) * world / (float(t[1]) * 1e-3)
    if cpu is not None:
        # parity: every pair's count against the CPU port over ALL shards of this rank (IntersectionCount form), then the executor-path timing
        want, _ = cpu.pairs(frags, shards, 1, materialise=False, rows_a=rows_a, rows_b=rows_b)
        if world > 1:                    # (the GPU counts are already merged across ranks by the library: fused exchange / ncclAllReduce)
            t = torch.tensor(np.asarray(want, dtype=np.int64), device="cuda")
            dist.all_reduce(t)
            want = t.cpu().numpy().astype(np.uint64)
        rec["parity_ok"] = bool(np.array_equal(got, want) and np.array_equal(got_single, want))
        rec["counts_sum"] = int(got.sum())
        if world == 1:
            _, ptimes = cpu.pairs(frags, shards, 3, materialise=True, rows_a=rows_a, rows_b=rows_b)
            psec = float(np.median(ptimes))
            rec["cpu_baseline"] = {"value": n_pairs * len(shards) / psec, "unit": "set-ops/s", "cores": cpu.threads, "kind": "port", "ms": psec * 1e3,
                                   "sample": "the %d pairs over all %d shards, 3 reps, median; executor path (Row.Intersect materialises, Count sums N)" % (n_pairs, len(shards))}
    return rec


def north_star(h, idx, fld, shards, cpu, frags, peak, world, dist, torch, steps):
    """BASELINE configs[4] at its acceptance point (1 %, 1 B columns per GPU)"""
    return pair_record(h, idx, fld, shards, PAIRS_A, PAIRS_B, "1 % density (uniform)", "north_star", cpu, frags, peak, world, dist, torch, steps)


SWEEP_POINTS = [(0.0001, 0, 8), (0.001, 0, 8), (0.1, 0, 2), (0.5, 0, 2), (0.01, 1, 8), (0.2, 1, 2)]   # (density, generator mode, row pairs); 1 % uniform = north_star


def density_sweep(h, idx, rank, S, cpu, peak, world, dist, torch, steps):
    """BASELINE configs[4]: the density sweep around the acceptance point (array / bitmap / run container mixes), on every rank's own
    shard range — at N GPUs this is the sweep `at 1, 2, 4, 8 GPUs` the north star asks for.  One field per point in the headline's
    context (same communicator); each point is parity-checked against the CPU port like the north-star record."""
    from featurebase_b200 import datagen as D, executor as X
    shards = np.arange(rank * S, (rank + 1) * S, dtype=np.uint64)
    out = []
    for k, (p, mode, n_pairs) in enumerate(SWEEP_POINTS):
        fld = idx.create_field("d%d" % k)
        rows = list(range(2 * n_pairs))
        bulk = D.fragments(40 + k, shards, rows, p, mode=mode, mean_run=64.0)
        h.ctx.load_fragments(idx.id, fld.id, X.VIEW_STANDARD, shards, bulk.buf, bulk.offsets)
        h.ctx.commit()
        frags = cpu.fragments(bulk, S) if cpu is not None else None
        label = "%g %% density (%s)" % (p * 100, "uniform" if mode == 0 else "clustered, mean run 64")
        rec = pair_record(h, idx, fld, shards, rows[0::2], rows[1::2], label, "density_sweep_%d" % k, cpu, frags, peak, world, dist, torch, max(steps // 2, 8))
        rec.update({"density": p, "generator": "uniform" if mode == 0 else "clustered"})
        out.append(rec)
        del bulk, frags
    return out


def config3(cpu, peak, steps, local):
    """BASELINE configs[2]: BSI Count(Row(v > k)), 10 M records, 32-bit values; 4 fields rotated so that the planes exceed L2"""
    from featurebase_b200 import datagen as D, executor as X, pql
    n_rec, nf = 10_000_000, 4
    n_sh = (n_rec + SW - 1) // SW
    shards = np.arange(n_sh, dtype=np.uint64)
    h = X.Holder(device=local)
    idx = h.create_index("b3", track_existence=False)
    ex = X.Executor(h)
    keep = []
    for k in range(nf):
        idx.create_field(f"v{k}", "int", min=0, max=(1 << 32) - 1)
        for s in range(n_sh):
            data = D.bsi_fragment(20 + k, s, min(SW, n_rec - s * SW), 32, 0, (1 << 32) - 1)
            h.import_roaring("b3", f"v{k}", X.VIEW_BSI, s, data)
            if k == 0:
                keep.append(data)
    h.ctx.commit()
    kval = 1 << 31
    progs = [ex._bitmap_call(idx, pql.parse(f"Row(v{k} > {kval})")[0]) for k in range(nf)]
    res = {}

    def step(i):
        res[i % nf] = h.ctx.count(idx.id, progs[i % nf], shards)

    ms, ms_min, wall = timed_calls(h.ctx, step, max(steps, 4 * nf), nf)
    LAST_OUTPUTS["config3_counts"] = np.array([res[k] for k in range(nf)], dtype=np.uint64)     # field k's last timed count
    pay, nc = h.ctx.rows_payload_bytes(idx.id, idx.fields["v0"].id, X.VIEW_BSI, shards, None)
    algo = pay + 16 * nc + 8
    rec = {"query": "Count(Row(v > 2^31)), 10,000,000 records, 32-bit int field", "kernel": "eval_wordpar_kernel", "ms": ms, "ms_min": ms_min, "e2e_ms": wall,
           "records_per_sec": n_rec / (ms * 1e-3), "algorithmic_bytes": int(algo), "gbs": algo / (ms * 1e-3) / 1e9, "frac": algo / (ms * 1e-3) / 1e9 / peak,
           "note": "algorithmic bytes = all 34 planes of the field (upper bound: the sweep stops early when the predicate saturates); 4 fields rotated (170 MB > L2)", "count": int(res[0])}
    if cpu is not None:
        frags = [cpu.O.Bitmap.from_bytes(d) for d in keep]
        want, secs = None, []
        for _ in range(3):
            want, s = cpu.O.bench_range_count(cpu.pool, frags, shards, ">", 32, kval)
            secs.append(s)
        rec["parity_ok"] = bool(want == res[0])
        sec = float(np.median(secs))
        rec["cpu_baseline"] = {"value": n_rec / sec, "unit": "records/s", "cores": min(cpu.threads, n_sh), "kind": "port", "ms": sec * 1e3,
                               "sample": "all 10 shards (one worker per shard: the reference maps per shard), 3 reps, median; fragment.rangeOp + Count"}
    h.ctx.close()
    return rec


def config4(cpu, peak, steps, local, rank, world, dist, torch, uid_fn):
    """BASELINE configs[3]: GroupBy(Rows(a), Rows(b)) 256 x 256 over 100 M records / 4096 shards: 512 shards per GPU (weak), the
    512 KiB count tensor summed with ncclAllReduce when N > 1"""
    from featurebase_b200 import datagen as D, executor as X
    S = 512
    p_rec = 100e6 / (4096 * SW)
    shards = np.arange(rank * S, (rank + 1) * S, dtype=np.uint64)
    h = X.Holder(device=local)
    idx = h.create_index("g4", track_existence=False)
    fa, fb = idx.create_field("a"), idx.create_field("b")
    fr_a, fr_b = [], []
    for s in shards:
        da, db = D.groupby_fragments(31, 32, int(s), p_rec, 256, 256)
        h.import_roaring("g4", "a", X.VIEW_STANDARD, int(s), da)
        h.import_roaring("g4", "b", X.VIEW_STANDARD, int(s), db)
        fr_a.append(da)
        fr_b.append(db)
    h.ctx.commit()
    if world > 1:
        h.ctx.comm_init(world, rank, uid_fn(h.ctx))
    rows = list(range(256))
    res = {}

    def step(i):
        res[0] = h.ctx.groupby(idx.id, [fa.id, fb.id], [0, 0], [rows, rows], shards)

    ms, ms_min, wall = timed_calls(h.ctx, step, max(steps, 10), 3)
    LAST_OUTPUTS["config4_groupby"] = np.asarray(res[0])
    if world > 1:
        t = torch.tensor([ms, wall], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, wall = float(t[0]), float(t[1])
    pa, na = h.ctx.rows_payload_bytes(idx.id, fa.id, 0, shards, None)
    pb, nb = h.ctx.rows_payload_bytes(idx.id, fb.id, 0, shards, None)
    algo = pa + pb + 16 * (na + nb) + 8 * 65536
    total = int(np.asarray(res[0]).sum())
    rec = {"query": "GroupBy(Rows(a), Rows(b)) 256 x 256, %d shards per GPU (%d in all), ~24.4 k records per shard" % (S, S * world), "kernel": ("groupby_shard_kernel" if os.environ.get("FBGPU_GROUPBY_HASH") else "groupby_direct_kernel"),
           "ms": ms, "ms_min": ms_min, "e2e_ms": wall, "records": total, "records_per_sec": total / (ms * 1e-3), "group_counts_per_sec": 65536 * S * world / (ms * 1e-3),
           "algorithmic_bytes_per_gpu": int(algo), "payload_bytes_per_gpu": int(pa + pb), "gbs": algo / (ms * 1e-3) / 1e9, "frac": algo / (ms * 1e-3) / 1e9 / peak,
           "count_merge": "ncclAllReduce(uint64, sum) of the 65536-entry tensor" if world > 1 else "none (one GPU)",
           "note": "ms = CUDA events around this rank's kernels (max over ranks); e2e_ms includes the all-reduce and the D2H of the tensor"}
    if cpu is not None:
        # parity: the FULL tensor against the CPU port over every shard of this rank (groupByIterator nested loop), summed over ranks
        fa_b = [cpu.O.Bitmap.from_bytes(d) for d in fr_a]
        fb_b = [cpu.O.Bitmap.from_bytes(d) for d in fr_b]
        want, sec = cpu.O.bench_groupby(cpu.pool, [fa_b, fb_b], shards, [rows, rows])
        if world > 1:
            t = torch.tensor(want.astype(np.int64), device="cuda")
            dist.all_reduce(t)
            want = t.cpu().numpy().astype(np.uint64)
        rec["parity_ok"] = bool(np.array_equal(np.asarray(res[0]).reshape(-1), want))
        if world == 1:
            rec["cpu_baseline"] = {"value": total / sec, "unit": "records/s", "cores": cpu.threads, "kind": "port", "ms": sec * 1e3,
                                   "sample": "all %d shards of this GPU's share, 1 rep; groupByIterator nested loop (65,536 intersectionCount calls per shard)" % S}
    h.ctx.close()
    return rec


def dump_outputs(path):
    """LAST_OUTPUTS as DIR/<name>.npy.  Every value is a count below 2^53, so float64 holds it exactly; all of them together
    are under 1 MB."""
    os.makedirs(path, exist_ok=True)
    for name, arr in LAST_OUTPUTS.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(arr, dtype=np.uint64).astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20, help="timed steps of the headline query")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--shards-per-gpu", type=int, default=1024)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU port (parity check and cpu_baseline records)")
    ap.add_argument("--no-extras", action="store_true", help="headline only (skip the north_star / config3 / config4 sub-records)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the density_sweep sub-record (six more fields are generated and loaded)")
    ap.add_argument("--extras", default="north_star,density_sweep,config3,config4", help="which sub-records to produce (comma list)")
    ap.add_argument("--reduce", default="p2p", choices=["p2p", "nccl"], help="N>1: fused peer-memory Count merge (default) or ncclAllReduce")
    ap.add_argument("--cold", action="store_true", help="also time fragment upload + query (e2e_cold_load)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what each timed query returned in its last timed step to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    if int(os.environ.get("LOCAL_RANK", "0")) == 0:
        import __graft_entry__
        __graft_entry__.build()          # no-op when libfbgpu.so / datagen / oracle are up to date

    import torch
    import torch.distributed as dist
    from featurebase_b200 import executor as X
    from featurebase_b200 import pql

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # the in-kernel wait of the fused Count merge is bounded (default 2 s, then FBGPU_E_COMM); the ranks of this script do seconds of host
    # work between collective queries while sharing the host cores, so the bound is widened here — it stays a bound (read when a context is created)
    os.environ.setdefault("FBGPU_P2P_TIMEOUT_MS", "20000")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()                   # rank 0 has finished building before the others load the library

    # ---- synthetic shard batch of this rank: contiguous shard range [rank*S, (rank+1)*S)  (SURVEY §8e)
    S = args.shards_per_gpu
    shards = np.arange(rank * S, (rank + 1) * S, dtype=np.uint64)
    t0 = time.time()
    bulk = gen_headline(shards)
    t_gen = time.time() - t0
    h = X.Holder(device=local)
    idx = h.create_index("i", track_existence=False)
    fld = idx.create_field("f")
    ex = X.Executor(h)
    t0 = time.time()
    h.ctx.load_fragments(idx.id, fld.id, X.VIEW_STANDARD, shards, bulk.buf, bulk.offsets)
    h.ctx.commit()
    t_load = time.time() - t0
    idx.shards.update(int(s) for s in shards)

    def new_uid(ctx):
        uid = [ctx.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        return uid[0]

    if world > 1:   # library-owned NCCL communicator for the count all-reduce
        h.ctx.comm_init(world, rank, new_uid(h.ctx))
        if args.reduce == "p2p":   # fused Count merge over NVLink peer memory (mailboxes mapped through CUDA IPC)
            ok = 1
            try:
                handles = [None] * world
                dist.all_gather_object(handles, h.ctx.comm_p2p_handle())
                h.ctx.comm_p2p_open(world, rank, handles)
            except Exception as e:  # noqa: BLE001 — e.g. a peer that cannot be IPC-mapped: every rank falls back together
                print(f"[rank {rank}] peer-memory merge unavailable ({e}); using ncclAllReduce", file=sys.stderr)
                ok = 0
            flag = torch.tensor([ok], device="cuda")
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            if int(flag.item()) == 0:
                if ok:
                    h.ctx.comm_p2p_disable()
                args.reduce = "nccl"
            dist.barrier()             # every rank has opened (and cleared) its mailbox before the first exchange
    ops = ex._bitmap_call(idx, pql.parse(query_text())[0].children[0])
    payload, n_cont = h.ctx.rows_payload_bytes(idx.id, fld.id, X.VIEW_STANDARD, shards, ROWS_A + ROWS_B)
    algo_bytes = payload + 16 * n_cont + 8                       # SURVEY §8d: payload + 16 B/descriptor + 8 B count
    h2d_bytes = 48 * len(ops) + 8 * len(shards)                  # fbgpu_op program + shard list (host buffers)
    ops = X.L.ops_array(ops)                                     # marshal the program once (host memory; still copied H2D by every call)
    shards = np.ascontiguousarray(np.asarray(shards, dtype=np.uint64))

    def step():
        return h.ctx.count(idx.id, ops, shards)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        expect = step()
    c0 = h.ctx.counters()["kernel_launches"]
    sampler = ClockSampler(local)
    sampler.start()
    sync_all()
    kernel_ms = []
    t_begin = time.perf_counter()
    for _ in range(args.steps):
        got = step()
        kernel_ms.append(h.ctx.counters()["last_query_gpu_ms"])   # CUDA events on the library's launching stream
        assert got == expect
    sync_all()
    wall = time.perf_counter() - t_begin
    LAST_OUTPUTS["headline_count"] = np.array([got], dtype=np.uint64)
    launches = h.ctx.counters()["kernel_launches"] - c0
    kms = float(np.mean(kernel_ms))
    # max over ranks (device time of the kernels; wall time of the C-ABI calls)
    if world > 1:
        t = torch.tensor([kms, wall], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        kms, wall = float(t[0]), float(t[1])
    # nvidia-smi cannot sample faster than ~10 Hz; when the timed region was shorter than that, keep the identical
    # step running (untimed; the SAME number of steps on every rank, the step contains a collective) until the sampler
    # has seen the GPU under this load, and say so
    probe_note = None
    if wall < 0.5:
        for _ in range(int(0.7 / max(wall / args.steps, 1e-5)) + 1):
            step()
        probe_note = "timed region %.0f ms < sampler period: clocks sampled over the timed region plus about 0.7 s of the identical step" % (wall * 1e3)
    clocks = sampler.stop()
    if probe_note:
        clocks["note"] = probe_note
    total_shards = S * world
    set_ops = SET_OPS_PER_SHARD * total_shards
    value = set_ops / (kms * 1e-3)
    e2e_ms = wall / args.steps * 1e3
    peak, peak_src = measured_peaks()
    achieved = algo_bytes / (kms * 1e-3) / 1e9
    traffic, traffic_note = None, "no ncu capture of this build under profiles/ (profiles/traffic.json is keyed by the kernel source hash)"
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of eval_kernel from an `ncu --set full` capture of THIS source state
        import hashlib
        src_hash = hashlib.sha1(open(os.path.join(ROOT, "featurebase_b200", "csrc", "kernels.cuh"), "rb").read()).hexdigest()[:16]
        tj = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))["eval_kernel"]
        if tj.get("kernels_cuh_sha1_16") == src_hash:
            traffic, traffic_note = tj["dram_bytes_per_launch"], "ncu --set full capture of this kernel source (profiles/traffic.json)"
        else:
            traffic_note = "profiles/traffic.json was captured on another kernel source (%s); not reported" % tj.get("kernels_cuh_sha1_16")
    except Exception:
        pass

    cold = None
    if args.cold and rank == 0:
        h2 = X.Holder(device=local)
        i2 = h2.create_index("i", track_existence=False)
        f2 = i2.create_field("f")
        t0 = time.perf_counter()
        h2.ctx.load_fragments(i2.id, f2.id, X.VIEW_STANDARD, shards, bulk.buf, bulk.offsets)
        n = h2.ctx.count(i2.id, ops, shards)
        cold = {"ms": (time.perf_counter() - t0) * 1e3, "h2d_bytes": int(bulk.offsets[-1]), "note": "parse + stage + H2D of every fragment, then the query"}
        assert n == expect or world > 1
        h2.ctx.close()

    # ---- parity at the BASELINE size, visible to the driver: the CPU port counts the same query over EVERY shard of every rank
    cpu, frags, parity, cpu_rec = None, None, None, None
    if not args.no_cpu_baseline:
        cpu = CpuArm()
        frags = cpu.fragments(bulk, S)
        if world == 1:
            cpu.calibrate(frags, shards)
        cnt, times = cpu.headline(frags, shards, 5 if world == 1 else 1)
        want = int(cnt)
        if world > 1:
            t = torch.tensor([want], device="cuda", dtype=torch.int64)
            dist.all_reduce(t)
            want = int(t.item())
        parity = {"parity_ok": bool(want == int(expect)), "cpu_count": want, "gpu_count": int(expect),
                  "what": "Count of the headline query over all %d shards: CPU port (every rank its own shards, summed) vs the GPU result after the cross-GPU merge" % total_shards}
        if world == 1:
            sec = float(np.median(times))
            cpu_rec = {"value": SET_OPS_PER_SHARD * S / sec, "unit": "set-ops/s", "cores": cpu.threads, "kind": "port", "ms": sec * 1e3, "calibration": cpu.calibration,
                       "sample": f"all {S} shards x 5 reps (median {sec * 1e3:.1f} ms); " + cpu.note}

    extras = {}
    want = set() if args.no_extras else set(args.extras.split(","))
    if args.no_sweep:
        want.discard("density_sweep")
    if "north_star" in want:
        extras["north_star"] = north_star(h, idx, fld, shards, cpu, frags, peak, world, dist, torch, args.steps)
    frags = None
    if "density_sweep" in want:
        extras["density_sweep"] = density_sweep(h, idx, rank, S, cpu, peak, world, dist, torch, args.steps)
    h.ctx.close()
    del bulk
    if "config3" in want and rank == 0 and world == 1:
        extras["config3"] = config3(cpu, peak, args.steps, local)
    if "config4" in want:
        extras["config4"] = config4(cpu, peak, args.steps, local, rank, world, dist, torch, new_uid)

    if rank == 0:
        line = {
            "metric": "set_ops_per_sec", "value": value, "unit": "set-ops/s", "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": kms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64/u16 integer", "data": "synthetic",
            "config": config_record(S, world, payload, args.reduce),
            "array_payload_order": "sorted (FBGPU_ARRAY_SORTED)" if os.environ.get("FBGPU_ARRAY_SORTED") else "bank-striped (default)",
            "count_rows_per_sec": total_shards / (kms * 1e-3), "columns_per_sec": total_shards * SW / (kms * 1e-3),
            "check_count": int(expect),
            "e2e": {"value": set_ops / (e2e_ms * 1e-3), "unit": "set-ops/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 8,
                    "note": "fbgpu_count() through the C ABI from host buffers (program + shard list H2D, count D2H) with fragments resident in HBM, wall clock"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "kernel": "eval_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_note": traffic_note, "algorithmic_bytes_per_launch": int(algo_bytes), "peak_source": peak_src,
                         "timing": "CUDA events on the library's launching stream around the kernel, mean over the timed steps"},
            "setup": {"datagen_s": t_gen, "load_commit_s": t_load, "payload_bytes_per_gpu": int(payload), "containers": int(n_cont)},
        }
        if parity:
            line.update(parity)
        if cpu_rec:
            line["cpu_baseline"] = cpu_rec
        if cold:
            line["e2e_cold_load"] = cold
        line.update(extras)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs)
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
