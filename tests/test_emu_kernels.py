"""The shipped kernels, interpreted on the CPU (tests/emu/): kernel LOGIC checked without a GPU.

tests/emu/ compiles a scratch copy of the library's own sources (fbgpu.cu + kernels.cuh, launches / `extern __shared__` /
inline PTX rewritten mechanically) with g++ against a stand-in <cuda_runtime.h> that runs every CUDA thread as a fibre, and the
gpu-marked parity tests are then re-run against that library in a child process.  This is test infrastructure: the product
never loads it (featurebase_b200/lib.py loads libfbgpu.so; FBGPU_LIB is the tuning-variant override the child uses), it
proves nothing about speed, memory-model races or the PTX the rewrites replace, and the device run stays the parity gate.
What it does give: the scatter / probe / program-loop / group-by code paths written after the round's GPU budget was spent
(and the opt-in ones: sorted array order, thread-per-row GroupBy, the unrolled word-parallel loop) have executed, statement
by statement, against the oracle and the reference's goldens.

Default run: everything gpu-marked except the staged (TMA) kernel and the bodies that take a minute or more each when
interpreted (≈1.5 min in all).  FBGPU_EMU_FULL=1 adds those: the 1024-shard property tests, the reference's 638 x 9
combination table (in both array orders), Percentile, the random aggregates (≈9 min)."""
import hashlib
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
EMU = os.path.join(HERE, "emu")
sys.path.insert(0, EMU)

FULL = bool(os.environ.get("FBGPU_EMU_FULL"))


def emu_lib(defines=(), flags=()):
    """build (once per source state) the interpreted library for the given -D list (+ extra compiler flags)"""
    import make_emu_source
    csrc = os.path.join(ROOT, "featurebase_b200", "csrc")
    srcs = [os.path.join(csrc, n) for n in sorted(os.listdir(csrc))] + [os.path.join(EMU, "cuda_runtime.h"), os.path.join(EMU, "make_emu_source.py"),
                                                                          os.path.join(ROOT, "include", "fbgpu.h")]
    h = hashlib.sha1()
    for p in srcs:
        h.update(open(p, "rb").read())
    h.update(" ".join(list(defines) + list(flags)).encode())
    out_dir = os.path.join(EMU, "_build", h.hexdigest()[:16])
    lib = os.path.join(out_dir, "libfbgpu_emu.so")
    if not os.path.exists(lib):
        make_emu_source.main(out_dir)
        cmd = ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-I", EMU, "-o", lib + ".tmp", os.path.join(out_dir, "fbgpu.cpp"), "-ldl", "-lpthread"]
        cmd += ["-D" + d for d in defines] + list(flags)
        subprocess.check_call(cmd)
        os.replace(lib + ".tmp", lib)
    return lib


def run_on_emulator(args, env=None, defines=(), timeout=1500):
    e = dict(os.environ, FBGPU_LIB=emu_lib(defines), FBGPU_TEST_ON_EMULATOR="1", **(env or {}))
    e.pop("FBGPU_EMU_FULL", None)
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider"] + args, cwd=ROOT, env=e,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=timeout)
    tail = "\n".join(r.stdout.splitlines()[-25:])
    assert r.returncode == 0, tail
    assert " passed" in tail and " failed" not in tail, tail
    return tail


NOT_HUGE = "not STAGED"                            # the staged kernel is TMA / mbarrier PTX: device only
SLOW = " and not full_size and not container_combinations and not sorted_order_set_ops and not percentile and not aggregates_random"      # a minute or more each when interpreted


def test_default_kernels_parity():
    """eval / pair-count / row-count / group-by / word-parallel / canonical-emit kernels of the default build against the
    oracle: tests/test_gpu_parity.py and the executor goldens (FULL adds the reference's 638 x 9 combination table)"""
    run_on_emulator(["tests/test_gpu_parity.py", "tests/test_zz_gpu_executor_goldens.py", "-k", NOT_HUGE + ("" if FULL else SLOW)], timeout=3000)


def test_query_level_bodies_on_interpreted_kernels():
    """the query-level tests written after the GPU budget ran out (aggregates, RBF loader, Distinct, time views, GroupBy
    pass shapes, ...) — on a GPU box these are plain gpu tests"""
    run_on_emulator(["tests/test_zz_gpu_experimental.py", "-k", NOT_HUGE + " and not sorted_order" + ("" if FULL else SLOW)], timeout=3000)


def test_node_fan_out_and_merge():
    """fbgpu_node (all devices of one process behind one handle): routing by shard owner, per-device fan-out on worker threads,
    host merge of counts / vectors / Row images, concurrent callers — two contexts stand in for two devices"""
    run_on_emulator(["tests/test_gpu_node.py"], timeout=3000)


def test_sorted_array_order():
    """FBGPU_ARRAY_SORTED=1: the reference's sorted element order (the default is the bank-striped one) under every kernel that reads array payloads"""
    run_on_emulator(["tests/test_zz_gpu_experimental.py", "-k", "sorted_order and " + NOT_HUGE + ("" if FULL else SLOW)], env={"FBGPU_TEST_EXPERIMENTAL": "1"}, timeout=3000)


def test_groupby_thread_per_row_variant():
    """FBGPU_GROUPBY_FAST=1 (groupby_kernel<true>): the GroupBy goldens and parity tests, and the shapes built for its passes
    (tiny arrays -> thread-per-row; a bitmap row / a 40-element row -> fallback inside the same kernel; two chunks per side; filter)"""
    sel = "(groupby or various_queries) and not sorted_order" + ("" if FULL else " and not full_size")
    # FBGPU_GROUPBY_CTA=1: groupby_kernel for every unit (by default it only sees what groupby_direct_kernel declines)
    run_on_emulator(["tests/test_gpu_parity.py", "tests/test_zz_gpu_experimental.py", "-k", sel], env={"FBGPU_GROUPBY_FAST": "1", "FBGPU_GROUPBY_CTA": "1"})
    run_on_emulator(["tests/test_gpu_parity.py", "tests/test_zz_gpu_experimental.py", "-k", "groupby and not sorted_order and not full_size"], env={"FBGPU_GROUPBY_CTA": "1"})


def test_wordpar_loop_variants():
    """the word-parallel op loop (wp_machine.h) with its register operand ring (-DFBGPU_WP_REG_RING), a shallower cp.async ring, and the
    round-1 rotating-ring loop (-DFBGPU_WP_LEGACY_LOOP), on the BSI programs (the default build's cp.async ring runs in test_default_kernels_parity)"""
    run_on_emulator(["tests/test_gpu_parity.py", "-k", "bsi_range or bsi_uniform or FORCE_WORDPAR or bsi_diagonal"], defines=("FBGPU_WP_REG_RING", "FBGPU_WP_RING=3"), timeout=3000)
    run_on_emulator(["tests/test_gpu_parity.py", "-k", "bsi_range or bsi_uniform or FORCE_WORDPAR"], defines=("FBGPU_WP_ASYNC_DEPTH=3",), timeout=3000)
    run_on_emulator(["tests/test_gpu_parity.py", "-k", "bsi_range or bsi_uniform or FORCE_WORDPAR"], defines=("FBGPU_WP_LEGACY_LOOP",), timeout=3000)


@pytest.mark.parametrize("order", ["reverse", "random"])
def test_results_do_not_depend_on_thread_order(order):
    """the same parity tests with the interpreter handing the CPU to runnable threads in reverse / pseudo-random order
    between barriers (FBGPU_EMU_ORDER): a missing barrier between a producer and a consumer phase shows up as a
    different result under one of the orders"""
    if order == "reverse" and not FULL:
        pytest.skip("reverse order: FBGPU_EMU_FULL=1 (the default suite runs the pseudo-random order)")
    sel = NOT_HUGE + SLOW + " and not thread_safety and not bsi_diagonal"
    run_on_emulator(["tests/test_gpu_parity.py", "tests/test_zz_gpu_experimental.py", "-k", sel + " and not sorted_order"], env={"FBGPU_EMU_ORDER": order, "FBGPU_GROUPBY_FAST": "1"}, timeout=3000)
    if FULL:
        run_on_emulator(["tests/test_gpu_parity.py", "-k", "groupby or density_sweep or mixed_encoding"], env={"FBGPU_EMU_ORDER": order}, timeout=3000)
        run_on_emulator(["tests/test_zz_gpu_experimental.py", "-k", "sorted_order_density_sweep or sorted_order_bsi"], env={"FBGPU_EMU_ORDER": order, "FBGPU_TEST_EXPERIMENTAL": "1"}, timeout=3000)


@pytest.mark.parametrize("san", ["undefined", "address"])
def test_interpreted_library_under_sanitizers(san):
    """kernels and host code compiled with -fsanitize=undefined (shifts, signed overflow, misaligned vector accesses abort)
    or -fsanitize=address (out-of-bounds on `__shared__` statics — plain red-zoned globals in that build —, on host
    vectors and on thread stacks): the parity tests, the sorted order, the GroupBy variant, the threaded API test"""
    if not FULL:
        pytest.skip("sanitizer builds: FBGPU_EMU_FULL=1")
    flags = ("-O1", "-g", "-fsanitize=undefined", "-fno-sanitize-recover=undefined") if san == "undefined" else ("-O1", "-g", "-fsanitize=address")
    lib = emu_lib(defines=() if san == "undefined" else ("FBGPU_EMU_PLAIN_SHARED",), flags=flags)
    rt = subprocess.run(["g++", "-print-file-name=" + ("libubsan.so" if san == "undefined" else "libasan.so")], stdout=subprocess.PIPE, text=True).stdout.strip()
    base = dict(os.environ, FBGPU_LIB=lib, FBGPU_TEST_ON_EMULATOR="1", LD_PRELOAD=rt, UBSAN_OPTIONS="print_stacktrace=1:halt_on_error=1",
                ASAN_OPTIONS="detect_leaks=0:halt_on_error=1")
    base.pop("FBGPU_EMU_FULL", None)
    for extra, sel in (({}, NOT_HUGE + SLOW + " and not sorted_order"),
                       ({"FBGPU_ARRAY_SORTED": "1", "FBGPU_GROUPBY_FAST": "1", "FBGPU_TEST_EXPERIMENTAL": "1"}, "(sorted_order or groupby or density_sweep) and " + NOT_HUGE + SLOW)):
        r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu", "-p", "no:cacheprovider", "tests/test_gpu_parity.py", "tests/test_zz_gpu_experimental.py", "-k", sel],
                           cwd=ROOT, env=dict(base, **extra), stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=3000)
        assert r.returncode == 0 and " passed" in r.stdout, r.stdout[-3000:]


def test_bench_main_runs_against_interpreted_library():
    """bench.py's own main() (GPU arm) on 8 shards with torch.cuda's device calls stubbed (tests/emu/bench_shim.py): the JSON
    line carries every key of the contract and the count agrees with the oracle-checked value for this data; the timings are
    meaningless.  Guards edits to bench.py made while no device was reachable."""
    import json
    e = dict(os.environ, FBGPU_LIB=emu_lib())
    r = subprocess.run([sys.executable, os.path.join(EMU, "bench_shim.py"), "--steps", "2", "--warmup", "1", "--shards-per-gpu", "8", "--no-cpu-baseline", "--no-extras"],
                       cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
              "e2e", "gpu_launches", "clocks", "roofline"):
        assert k in d, k
    assert d["warmup"] >= 3 and d["gpu_launches"] == 2 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 8
    assert set(d["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and "NOT a valid bench size" in d["config"]["l2"]
    # the same query through the oracle-backed mirror
    sys.path.insert(0, ROOT)
    import bench
    from featurebase_b200 import datagen as D
    from oracle import oracle as O
    exp = 0
    for s in range(8):
        fr = O.Bitmap.from_bytes(D.fragment(bench.FIELD_SEED_ID, s, bench.ROWS_A + bench.ROWS_B, 0.01))
        a, b = O.Bitmap(), O.Bitmap()
        for rr in bench.ROWS_A:
            a = a.union(fr.row(rr, s))
        for rr in bench.ROWS_B:
            b = b.union(fr.row(rr, s))
        exp += a.intersect(b).count()
    assert d["check_count"] == exp > 0


def test_bench_sub_records_run_against_interpreted_library(tmp_path):
    """bench.py's north_star and density_sweep sub-records on 4 shards, CPU port included: every point's parity_ok (GPU arm's counts,
    single and batched, against the CPU port over all shards) must hold — these are the checks bench.py reports at full size.
    --dump-outputs writes the same counts as .npy files."""
    import json
    import numpy as np
    e = dict(os.environ, FBGPU_LIB=emu_lib())
    r = subprocess.run([sys.executable, os.path.join(EMU, "bench_shim.py"), "--steps", "2", "--warmup", "1", "--shards-per-gpu", "4", "--extras", "north_star,density_sweep",
                        "--dump-outputs", str(tmp_path)], cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=1500)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["parity_ok"] is True and d["north_star"]["parity_ok"] is True and d["north_star"]["counts_sum"] > 0
    assert len(d["density_sweep"]) == 6
    for rec in d["density_sweep"]:
        assert rec["parity_ok"] is True, rec["query"]
        assert rec["container_pair_types_pair0"] and "cpu_baseline" in rec
    kinds = set(k for rec in d["density_sweep"] for k in rec["container_pair_types_pair0"])
    assert {"array x array", "bitmap x bitmap"} <= kinds and any("run" in k for k in kinds), kinds
    out = {p.stem: np.load(p) for p in tmp_path.glob("*.npy")}
    names = {"headline_count"} | {"%s_%s" % (n, k) for n in ["north_star"] + ["density_sweep_%d" % i for i in range(6)] for k in ("single", "batched")}
    assert set(out) == names and all(a.dtype == np.float64 for a in out.values())
    assert out["headline_count"].tolist() == [d["check_count"]]
    assert out["north_star_batched"].shape == (32,) and out["north_star_batched"].sum() == d["north_star"]["counts_sum"]
    for i, rec in enumerate(d["density_sweep"]):
        assert np.array_equal(out["density_sweep_%d_single" % i], out["density_sweep_%d_batched" % i])
        assert out["density_sweep_%d_batched" % i].sum() == rec["counts_sum"]


def test_bench_sweep_runs_against_interpreted_library():
    """bench_sweep.py (configs 5 / 5b / 4 / X / R at 2 shards, one step) incl. its own checks against the oracle and the data
    generator — guards the script the round-2 first call runs; timings meaningless"""
    import json
    e = dict(os.environ, FBGPU_LIB=emu_lib())
    r = subprocess.run([sys.executable, "bench_sweep.py", "--configs", "5,4,X,R", "--shards", "2", "--groupby-shards", "2", "--steps", "1", "--densities", "0.01",
                        "--generators", "uniform,clustered", "--batched"], cwd=ROOT, env=e, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    rows = [json.loads(l) for l in r.stdout.strip().splitlines()]
    assert [str(d["config"]) for d in rows] == ["5", "5b", "5", "5b", "4", "X", "X", "X", "X", "X", "R", "R", "R"]


def test_interpreter_reports_divergent_barriers():
    """the interpreter's own checks: a barrier only part of a block reaches is reported (not silently passed), full-mask warp
    primitives see every lane, shared-memory reductions land where the 32-bit shared address says, and a read past the end of
    a device buffer faults"""
    src = os.path.join(EMU, "selftest.cpp")
    exe = os.path.join(EMU, "_build", "selftest")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-I", EMU, "-o", exe, src, "-lpthread"])
    assert subprocess.run([exe, "ok"], stdout=subprocess.PIPE, text=True).stdout.strip() == "selftest ok"
    r = subprocess.run([exe, "diverge"], stderr=subprocess.PIPE, text=True)
    assert r.returncode != 0 and "deadlock" in r.stderr
    r = subprocess.run([exe, "overrun"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
    assert r.returncode < 0 and "in bounds ok" in r.stdout and "not reached" not in r.stdout      # killed by SIGSEGV at the guard page
