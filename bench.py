#!/usr/bin/env python
"""bench.py — trace rows/sec proven (Fibonacci, BASELINE.json metric) on N B200s of one node.

A "step" is one full Machine::prove() of the workload (LDE + Keccak Merkle commits + LogUp perm trace
+ quotient + FRI opening), from traces to CBOR proof bytes.
  value  : whole-job rows/s with the traces already resident in HBM (vgpu_prove_device)
  e2e    : the same metric through the reference-facing C-ABI call with HOST buffers
           (vgpu_prove: H2D of the pinned traces + D2H of the proof inside the timed region)
  N > 1  : ONE proof per step split across the N GPUs (row shards after one peer-store exchange over NVLink,
           sub-roots all-gathered): value = rows of that proof / max-over-ranks time ("scaling": "strong");
           the N-independent-proofs figure is reported beside it under "replicas".
  --impl reference : the CPU restatement of the reference prover (oracle/, all host threads) on a
           bounded sample of the same workload; rank 0 only.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True      # the benchmark leaves the tree it runs from as it found it
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# torchrun pins OMP_NUM_THREADS to 1 for every rank; the host witness generator (and the CPU arm's trace generation) use OpenMP.
# Give each rank its share of the host cores — before anything loads the OpenMP runtime.
if os.environ.get("OMP_NUM_THREADS") == "1" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
    os.environ["OMP_NUM_THREADS"] = str(max(1, (os.cpu_count() or 1) // int(os.environ.get("LOCAL_WORLD_SIZE", os.environ["WORLD_SIZE"]))))

# CPU arm: keep the oracle's threads on neighbouring cores of one socket (measured on the 2 x 32-core host: 1.65 -> 1.53 s per 2^18-row proof).
if "reference" in sys.argv:
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")

FIB_N = {22: 599183, 20: 149794, 18: 37447, 17: 9360 * 2, 16: 9360, 15: 2339, 12: 582, 8: 25}   # log2(CPU rows) -> n (cycles = 17 + 7n)


def fib_n_for_log_rows(log_rows):
    # largest n with 17 + 7n <= 2^log_rows
    return ((1 << log_rows) - 17) // 7


_JSON_OUT = None


def emit(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic_ratio(kernel):
    """DRAM bytes moved / algorithmic bytes for one kernel class, from the committed `ncu --set full` raw pages:
    ntt_pass_kernel: profiles/r02_ntt_v7_raw.csv (the shipping kernel: 8 launches over a 2^22 x 16 matrix, 8 B per element per launch);
    compress_layer_kernel: profiles/r02_compress_raw.csv (the shipping kernel: tree layers of 2^24 .. 2^21 nodes, 96 B per node)."""
    import csv

    spec = {"ntt_pass_kernel": ("r02_ntt_v7_raw.csv", "ntt_pass", lambda gx, gy: 8.0 * gx * gy * (1 << 14)),      # a 2^14-element tile per CTA
            "compress_layer_kernel": ("r02_compress_raw.csv", "compress_layer", lambda gx, gy: 96.0 * gx * 128)}  # a node per thread
    if kernel not in spec:
        return None, None
    fname, tag, alg_bytes = spec[kernel]
    path = os.path.join(ROOT, "profiles", fname)
    try:
        rows = list(csv.reader(open(path)))
        hdr, units = rows[0], rows[1]
        ir, iw, ig, ik = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum"), hdr.index("Grid Size"), hdr.index("Kernel Name")
        scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}
        tot, alg = 0.0, 0.0
        for r in rows[2:]:
            if tag not in r[ik]:
                continue
            tot += float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]]
            gx, gy = [int(v) for v in r[ig].strip("()").split(",")[:2]]
            alg += alg_bytes(gx, gy)
        return tot / alg, os.path.relpath(path, ROOT)
    except Exception:
        return None, None


def aggregate_throughput(dist, rows_local, ms_local, device=None, sum_rows=True):
    """Whole-job rows/s: rows / max-over-ranks time.  sum_rows: every rank proves its own trace (replicas); otherwise all
    ranks work on the SAME proof and the rows count once."""
    import torch

    t = torch.tensor([float(ms_local)], dtype=torch.float64, device=device)
    r = torch.tensor([float(rows_local)], dtype=torch.float64, device=device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if sum_rows:
            dist.all_reduce(r, op=dist.ReduceOp.SUM)
    return float(r.item()) / (float(t.item()) / 1000.0), float(t.item())


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.stop_flag, self.th = index, [], False, None

    def _run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.15)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag = True
        if self.th:
            self.th.join(timeout=6)
        sm = sorted(int(r[0]) for r in self.rows if r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if r[1].isdigit()] or [0])
        reasons = []
        for name, col in (("hw_slowdown", 3), ("hw_thermal_slowdown", 4), ("sw_thermal_slowdown", 5), ("sw_power_cap", 6)):
            if any(len(r) > col and r[col].lower().startswith("active") for r in self.rows):
                reasons.append(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons, "samples": len(self.rows)}


_HOST = None


def host_cpus():
    """What the host really grants this process: logical CPUs, the scheduler affinity mask, and the container's CPU quota (cgroup
    v2 cpu.max / v1 cfs_quota) — os.cpu_count() alone over-reports inside a limited container, and OpenMP threads beyond the
    quota only get throttled."""
    global _HOST
    if _HOST is not None:
        return _HOST
    info = {"logical": os.cpu_count() or 1}
    try:
        info["affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity"] = info["logical"]
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    info["cgroup_quota_cpus"] = quota
    try:
        info["loadavg_1m"] = os.getloadavg()[0]
    except Exception:
        pass
    usable = min(info["logical"], info["affinity"])
    if quota:
        usable = max(1, min(usable, int(quota + 0.5)))
    info["usable"] = usable
    _HOST = info
    return info


def thread_candidates(usable):
    """Thread counts the CPU arm tries on the sample itself: beyond 64 the oracle's short parallel regions oversubscribe
    (measured on the 128-CPU box: 3.4 s at 16 / 32, 4.8 s at 64, 51 s at 128 threads for the same 2^18-row proof)."""
    return sorted({max(1, min(usable, c)) for c in (16, 32, 64)})


def _tracegen_to_files(workload, log_rows, out_prefix):
    """Child-process entry (python bench.py --tracegen ...): the witness generator lives in the product library, the
    reference arm must not load it — so the traces reach the reference process as .npy files."""
    import numpy as np

    t, _, _ = build_traces(workload, log_rows)
    for i, m in enumerate(list(t.main) + list(t.preprocessed)):
        np.save("%s.%d.npy" % (out_prefix, i), np.ascontiguousarray(m))


def _load_trace_files(workload, log_rows):
    import numpy as np
    import shutil
    import tempfile

    # ~2.1 GB of traces at 2^22 CPU rows (Fibonacci); /dev/shm when it has the room (a container's default is 64 MB), else the temp dir
    need = int(2.6e9 * (1 << log_rows) / (1 << 22)) + (64 << 20)
    base = None
    try:
        st = os.statvfs("/dev/shm")
        if st.f_bavail * st.f_frsize > need:
            base = "/dev/shm"
    except OSError:
        pass
    d = tempfile.mkdtemp(prefix="vgpu_ref_", dir=base)
    try:
        prefix = os.path.join(d, "t")
        subprocess.run([sys.executable, os.path.abspath(__file__), "--tracegen", prefix, "--workload", workload, "--log-rows", str(log_rows)], check=True)
        mats = [np.load("%s.%d.npy" % (prefix, i)) for i in range(16)]
    finally:
        shutil.rmtree(d, ignore_errors=True)
    return mats[:14], mats[14:]


def _prefault(orc, log_rows):
    """A size that is proven ONCE would spend much of its time in first-touch page faults taken on one thread (measured: 28.0 s for the
    first 2^20-row proof of a process against 17.6 s for the second, 21.5 s of it kernel time); the heap is grown and touched on all
    threads first (about 1 s per 7 GB), which is what the warm-up steps do for the sample size.  Skipped when memory is short."""
    need = int(7.4e9 * (1 << log_rows) / (1 << 20))
    try:
        avail = 0
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable:"):
                avail = int(ln.split()[1]) * 1024
        if avail > 2 * need:
            orc.prefault_heap(need)
    except Exception:
        pass


def cpu_baseline_leg(workload, cbl):
    """`cpu_baseline` of the GPU arm's line: the oracle (CPU restatement of the reference prover) on a bounded sample of the
    workload, on the box's host cores.  The last thing the process does: the heap is kept and touched up front, so that the
    first candidate is not the one that pays for the page faults; thread sweep on the sample itself, then the fastest count once
    more (best of its two runs)."""
    from valida_b200 import build as vbuild
    import oracle_binding

    vbuild.build_oracle()
    orc = oracle_binding.Oracle()
    tb, _, _ = build_traces(workload, cbl)
    host = host_cpus()
    cores = host["logical"]
    orc.tune_allocator()
    _prefault(orc, cbl)
    best, sweep = None, {}
    for th in thread_candidates(host["usable"]) + [None]:
        if th is None:
            th = best[1]
        orc.set_threads(th)
        t0 = time.perf_counter()
        ref = orc.prove(tb.main, tb.preprocessed, debug_checks=False)
        dt = time.perf_counter() - t0
        del ref
        sweep.setdefault(str(th), []).append(dt)
        if best is None or dt < best[0]:
            best = (dt, th)
    return {"value": tb.main[0].shape[0] / best[0], "unit": "rows/s", "cores": best[1], "kind": "port",
            "sample": "%s at 2^%d CPU rows, one full oracle prove, %.1f s, %d OpenMP threads (fastest of a sweep on this size) on %d host cores"
                      % (workload, cbl, best[0], best[1], cores), "host": host, "thread_sweep_s": sweep}


def run_reference(args, rank):
    """Reference arm: the CPU restatement of the reference prover (oracle/, all the host threads it can use) proving a
    bounded sample of the arm's workload per step.  The warm-up steps double as the thread sweep — on the SAMPLE ITSELF, so the
    timed steps run at the thread count that proved this very size fastest — and one extra proof at a larger size shows how
    the per-row cost moves with the size (the extrapolation to the full workload is then visible, not assumed)."""
    if rank != 0:
        return
    t_arm0 = time.perf_counter()
    from valida_b200 import build as vbuild          # build helper only: the product library is NOT loaded in this process
    import oracle_binding

    vbuild.build_oracle()
    orc = oracle_binding.Oracle()
    orc.tune_allocator()                             # freed vectors stay in the heap: no page faults on every re-allocation
    workload, full_log_rows = resolve_workload(args)
    log_rows = min(args.ref_log_rows, full_log_rows)
    main, prep = _load_trace_files(workload, log_rows)
    rows = main[0].shape[0]
    host = host_cpus()
    cores = host["logical"]
    cand = thread_candidates(host["usable"])
    sweep, times = {}, []
    threads = cand[-1]
    for i in range(args.warmup + args.steps):
        if i < args.warmup:
            threads_i = cand[i % len(cand)]
        else:
            if i == args.warmup and sweep:
                threads = min(sweep, key=lambda k: min(sweep[k]))
            threads_i = threads
        orc.set_threads(threads_i)
        t0 = time.perf_counter()
        pr = orc.prove(main, prep, debug_checks=False)
        dt = time.perf_counter() - t0
        del pr
        if i < args.warmup:
            sweep.setdefault(threads_i, []).append(dt)
        else:
            times.append(dt)
    total = sum(times)
    value = rows * len(times) / total
    sizes = {"2^%d" % log_rows: {"rows_per_s": value, "s_per_proof": total / len(times), "threads": threads, "proofs": len(times)}}
    del main, prep
    # one proof at each further size (by default 2^18 and the arm's full workload, 2^22): how the per-row cost moves with the size is then
    # measured, not extrapolated; a size that fails (memory, temp space) is recorded and changes nothing above
    for extra in [int(x) for x in str(args.ref_extra_log_rows).split(",") if x.strip() and int(x) > 0]:
        if extra > full_log_rows or extra == log_rows:
            continue
        # the whole arm is meant to end within a few minutes: a further size is skipped when its projected time (per-row cost of the
        # sample, with 50 % on top) would take the run past the budget
        projected = 1.5 * (total / len(times)) * (1 << extra) / (1 << log_rows)
        if time.perf_counter() - t_arm0 + projected > args.ref_budget_s:
            sizes["2^%d" % extra] = {"skipped": "projected %.0f s would pass the arm's time budget of %d s" % (projected, args.ref_budget_s)}
            continue
        try:
            m2, p2 = _load_trace_files(workload, extra)
            orc.set_threads(threads)
            _prefault(orc, extra)
            t0 = time.perf_counter()
            pr = orc.prove(m2, p2, debug_checks=False)
            dt = time.perf_counter() - t0
            del pr
            sizes["2^%d" % extra] = {"rows_per_s": m2[0].shape[0] / dt, "s_per_proof": dt, "threads": threads, "proofs": 1}
            del m2, p2
        except Exception as exc:   # noqa: BLE001
            sizes["2^%d" % extra] = {"error": "%s: %s" % (type(exc).__name__, exc)}
    full_key = "2^%d" % full_log_rows
    full_measured = full_key in sizes and "rows_per_s" in sizes[full_key]
    # BASELINE.json configs[0], the reference's own test: prove_fibonacci n = 25 (192 cycles; CPU chip 2^8 rows, mul chip floor 2^10)
    config1 = None
    try:
        m1, p1 = _load_trace_files("fibn25", 8)
        config1 = {"program": "fib n=25 (basic/tests/test_prover.rs:474-487): 192 cycles, CPU trace 2^8 rows"}
        for th in sorted({1, threads}):
            orc.set_threads(th)
            ts = []
            for _ in range(7):
                t0 = time.perf_counter()
                pr = orc.prove(m1, p1, debug_checks=False)
                ts.append(time.perf_counter() - t0)
                del pr
            config1["ms_per_proof_%d_threads" % th] = 1e3 * sorted(ts)[len(ts) // 2]
    except Exception as exc:   # noqa: BLE001
        config1 = {"error": "%s: %s" % (type(exc).__name__, exc)}
    # BASELINE.json configs[1] on the CPU: 2^20 x 64 NTT + inverse through the oracle's transform (natural order in and out; the
    # call copies the matrix in and out, which is inside the figure: ~0.5 GB of memcpy against 44 butterfly sweeps)
    config2 = None
    try:
        import ctypes
        import numpy as np

        hh, ww = 1 << 20, 64
        rr = np.arange(hh, dtype=np.uint64)[:, None]
        cc = np.arange(ww, dtype=np.uint64)[None, :]
        x = ((rr * 64 + cc) * 0x9E3779B1 % 2013265921).astype(np.uint32)          # SURVEY 8(d) config 2 input
        y = x.copy()
        u32p = ctypes.POINTER(ctypes.c_uint32)
        orc.set_threads(threads)
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            orc.L.orc_dft(y.ctypes.data_as(u32p), ctypes.c_uint64(hh), ctypes.c_uint64(ww), 0)
            orc.L.orc_dft(y.ctypes.data_as(u32p), ctypes.c_uint64(hh), ctypes.c_uint64(ww), 1)
            dt = time.perf_counter() - t0
            best = dt if best is None or dt < best else best
        config2 = {"workload": "2^20 x 64 NTT + iNTT (oracle, natural order in/out)", "ms_forward_plus_inverse": 1e3 * best, "threads": threads,
                   "achieved": 2 * 8.0 * hh * ww / best / 1e9, "unit": "GB/s", "bytes": "8*h*w per transform", "roundtrip_bit_exact": bool(np.array_equal(x, y))}
        del x, y
    except Exception as exc:   # noqa: BLE001
        config2 = {"error": "%s: %s" % (type(exc).__name__, exc)}
    sample = "%s at 2^%d CPU rows (one full prove per step; the arm's workload is 2^%d rows); %d OpenMP threads (fastest of %s in the warm-up steps, on this size) of %d host cores" % (
        workload, log_rows, full_log_rows, threads, cand, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * total / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": DTYPE, "data": "synthetic",
        "config": {"workload": workload_name(workload, full_log_rows), "sample": sample, "same_config": log_rows == full_log_rows,
                   "full_workload_measured_once": full_measured, "full_workload_rows_per_s": sizes[full_key]["rows_per_s"] if full_measured else None},
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "sizes": sizes, "thread_sweep_s": {str(k): min(v) for k, v in sweep.items()}, "host": host, "config1_prove_fibonacci_n25": config1, "config2_ntt": config2,
        "note": "the real reference (Rust + un-vendored Plonky3) cannot be built here; this is oracle/, the C++ restatement, OpenMP; rows/s at the measured sizes are in `sizes`",
    }
    emit(line)


METRIC = "trace rows/sec proven"
DTYPE = "u32 (BabyBear, 31-bit modular) + ext5"


def resolve_workload(args):
    """--workload fib22 | fib24 | config5 | fib | config5 (+ --log-rows) -> (family, log2 CPU rows)."""
    w = args.workload
    if w.startswith("fib") and w[3:].isdigit():
        return "fib", int(w[3:])
    if w == "config5":
        return "config5", args.log_rows
    return w, args.log_rows


def build_traces(workload, log_rows):
    """Host witness of the workload (Chip::generate_trace x14): (traces, CPU rows, description)."""
    import valida_b200 as vb

    program, what = workload_program(workload, log_rows)
    t = vb.run_program(program, initial_fp=0x1000)
    rows = t.main[0].shape[0]
    assert rows == 1 << log_rows, (rows, log_rows)
    return t, rows, what


def workload_program(workload, log_rows):
    import valida_b200 as vb

    if workload == "fib":
        n = fib_n_for_log_rows(log_rows)
        return vb.fib_program(n), "fib n=%d" % n
    if workload == "fibn25":       # BASELINE.json configs[0]: prove_fibonacci of basic/tests/test_prover.rs (n = 25: 192 cycles, 2^8 CPU rows)
        return vb.fib_program(25), "fib n=25"
    if workload == "config5":
        from programs import config5_program

        iters = ((1 << log_rows) - 8) // 15
        return config5_program(iters), "config5_program(%d)" % iters
    raise SystemExit("unknown workload %r" % workload)


def workload_name(workload, log_rows):
    if workload == "fib":
        return "Fibonacci 2^%d-row full prove (LDE+perm+quotient+FRI+Keccak Merkle), BasicMachine 14 chips, blowup 2, 40 queries" % log_rows
    return "multi-chip synthetic program (add, sub, lt family, and/or/xor, memory, range; SURVEY 8(d) config 5), 2^%d CPU rows, full prove, BasicMachine 14 chips, blowup 2, 40 queries" % log_rows


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="fib22", help="fib22 (BASELINE config 3, default) | fib24 (config 4) | config5 | fib / config5 with --log-rows")
    ap.add_argument("--log-rows", type=int, default=22, help="log2 of the CPU-chip trace height for --workload fib / config5")
    ap.add_argument("--ref-log-rows", type=int, default=20, help="bounded sample size of the CPU reference arm (one proof per step)")
    ap.add_argument("--ref-extra-log-rows", default="18,22", help="reference arm: one extra proof at each of these sizes (comma separated; 0 = none)")
    ap.add_argument("--ref-budget-s", type=int, default=300, help="reference arm: further sizes are skipped when they would take the run past this many seconds")
    ap.add_argument("--cpu-baseline-log-rows", type=int, default=18)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-replicas", action="store_true", help="N > 1: skip the independent-proofs-per-GPU figure")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (the CBOR proof, one byte per float32) to DIR/proof.npy")
    ap.add_argument("--tracegen", default=None, help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.tracegen:
        w, lr = resolve_workload(args)
        _tracegen_to_files(w, lr, args.tracegen)
        return

    host_cpus()      # read the affinity mask before an OpenMP runtime loads: with OMP_PROC_BIND set libgomp pins the initial thread to one place
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    # stdout carries exactly one JSON line.  Libraries print there too (NCCL's "NCCL version ..." banner comes out of
    # a C printf on rank 0), so file descriptor 1 is pointed at stderr for the whole run and the JSON line is written to
    # a private duplicate of the original stdout.
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import valida_b200 as vb
    from valida_b200 import build as vbuild

    if not os.path.exists(vb.lib_path):
        vbuild.build()
    torch.cuda.set_device(local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    # an explicit (non-default) torch stream: its handle is non-null, so the library enqueues on it and
    # torch.cuda.Event timings on this stream see the library's kernels
    stream = torch.cuda.Stream()
    torch.cuda.set_stream(stream)
    ctx = vb.Context(local_rank, stream=stream.cuda_stream)
    assert stream.cuda_stream != 0
    rc = np.zeros(480, dtype=np.uint32)
    # documented stand-in for the caller's Poseidon RNG (DESIGN.md): SplitMix64("valida"), 31-bit rejection sampling
    state, k, M = 0x76616C696461, 0, (1 << 64) - 1
    while k < 480:
        state = (state + 0x9E3779B97F4A7C15) & M
        z = state
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & M
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & M
        z ^= z >> 31
        c = z >> 33
        if c < vb.BABYBEAR_P:
            rc[k] = c
            k += 1
    cfg = vb.StarkConfig(ctx, rc)
    def watchdog():      # a rank that died leaves the others inside a collective, a kernel may never end: end the run instead of hanging the box
        time.sleep(1500)
        sys.stderr.write("bench.py: watchdog — the run did not finish within 1500 s\n")
        os._exit(3)

    threading.Thread(target=watchdog, daemon=True).start()
    if dist is not None:
        # N > 1: ONE proof per step, split across the ranks (row shards after one peer-store exchange; include/valida_b200.h)
        ctx.comm_init_from_torch()

    workload, log_rows = resolve_workload(args)
    t0 = time.perf_counter()
    traces, rows, what = build_traces(workload, log_rows)
    tracegen_s = time.perf_counter() - t0
    trace_bytes = sum(m.nbytes for m in traces.main) + sum(m.nbytes for m in traces.preprocessed)

    # pinned host copies for the e2e path; device-resident copies (this rank's row shards when the proof is split) for `value`
    pinned = []
    for m in list(traces.main) + list(traces.preprocessed):
        tt = torch.empty(m.shape, dtype=torch.int32, pin_memory=True)
        tt.numpy().view(np.uint32)[...] = m
        pinned.append(tt)

    class PinnedTraces:
        main = [p.numpy().view(np.uint32) for p in pinned[:14]]
        preprocessed = [p.numpy().view(np.uint32) for p in pinned[14:]]

    dm = [ctx.upload_rows(m) for m in traces.main]
    dp = [ctx.upload_rows(m) for m in traces.preprocessed]
    ctx.synchronize()
    # bytes a rank uploads per step on the e2e path: its rows of the tall traces, the short ones whole
    h2d_local = 0
    for m, d in zip(list(traces.main) + list(traces.preprocessed), dm + dp):
        h2d_local += d.local_rows()[1] * m.shape[1] * 4

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks / throttle reasons are sampled from the first warm-up step to the end of the timed region (the same load
    # throughout; one nvidia-smi query takes ~0.3 s, the timed region alone would see one or two samples)
    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(args.warmup):
        vb.prove_machine(cfg, traces, device_resident=(dm, dp))

    # ---- timed: device-resident, no instrumentation ----
    launches0 = ctx.launch_count
    ctx.comm_stats()
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        proof = vb.prove_machine(cfg, traces, device_resident=(dm, dp))
    ev1.record(stream)
    barrier()
    clocks = sampler.stop()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    comm = ctx.comm_stats()
    phases = vb.last_prove_phases(ctx)
    # one proof per step whatever N: rows proven = rows * steps, time = the slowest rank's
    value, ms_total_max = aggregate_throughput(dist, rows * args.steps, ms_total, device="cuda", sum_rows=False)
    if args.dump_outputs and rank == 0:
        # every rank of a split proof returns the same bytes; float32 holds each byte exactly
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "proof.npy"), np.frombuffer(proof, dtype=np.uint8).astype(np.float32))

    # ---- the same K steps again with a CUDA-event pair around every kernel launch (per-kernel roofline) ----
    ctx.set_kernel_timing(True)
    vb.prove_machine(cfg, traces, device_resident=(dm, dp))   # populates the event pool
    ctx.kernel_stats()
    barrier()
    ei0, ei1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ei0.record(stream)
    for _ in range(args.steps):
        vb.prove_machine(cfg, traces, device_resident=(dm, dp))
    ei1.record(stream)
    barrier()
    ms_instr = ei0.elapsed_time(ei1)
    kstats = ctx.kernel_stats()
    ctx.set_kernel_timing(False)

    # ---- timed: end to end through the host-buffer C-ABI call (every rank copies ITS rows of the pinned traces) ----
    vb.prove_machine(cfg, PinnedTraces)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        proof_e2e = vb.prove_machine(cfg, PinnedTraces)
    e1.record(stream)
    barrier()
    ms_e2e = e0.elapsed_time(e1)
    e2e_value, _ = aggregate_throughput(dist, rows * args.steps, ms_e2e, device="cuda", sum_rows=False)
    assert proof_e2e == proof
    h2d_total = h2d_local
    proofs_identical = True
    if dist is not None:
        tsum = torch.tensor([float(h2d_local)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tsum)
        h2d_total = float(tsum.item())
        import hashlib

        dig = int.from_bytes(hashlib.sha256(proof).digest()[:7], "big")
        tmin = torch.tensor([float(dig)], dtype=torch.float64, device="cuda"); tmax = tmin.clone()
        dist.all_reduce(tmin, op=dist.ReduceOp.MIN); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        proofs_identical = bool(tmin.item() == tmax.item())

    # ---- the same call from PAGEABLE caller memory (what a Rust Vec is), and from the same memory page-locked in place ----
    e2e_other = {}
    try:
        steps_p = min(args.steps, 3)
        def timed(label):
            vb.prove_machine(cfg, traces)
            barrier()
            p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            p0.record(stream)
            for _ in range(steps_p):
                pr = vb.prove_machine(cfg, traces)
            p1.record(stream)
            barrier()
            v, _ = aggregate_throughput(dist, rows * steps_p, p0.elapsed_time(p1), device="cuda", sum_rows=False)
            e2e_other[label] = {"value": v, "unit": "rows/s", "proof_equals": bool(pr == proof)}
        timed("pageable")
        t0 = time.perf_counter()
        for m in list(traces.main) + list(traces.preprocessed):
            ctx.host_register(m)
        e2e_other["register_s"] = time.perf_counter() - t0
        timed("registered_in_place")
        for m in list(traces.main) + list(traces.preprocessed):
            ctx.host_unregister(m)
    except Exception as exc:   # noqa: BLE001
        e2e_other["error"] = "%s: %s" % (type(exc).__name__, exc)

    # ---- from the PROGRAM to the proof: host interpreter -> logs -> device row fill (witness.cu) -> prove; beside it the host row fill ----
    with_witness = None
    try:
        program, _ = workload_program(workload, log_rows)
        best = None
        for _ in range(2):
            barrier()
            t0 = time.perf_counter()
            log = vb.run_program_log(program)
            t1 = time.perf_counter()
            wm, wp = log.witness_device(ctx)
            ctx.synchronize()
            t2 = time.perf_counter()
            proof_w = vb.prove_machine(cfg, traces, device_resident=(wm, wp))
            ctx.synchronize()
            t3 = time.perf_counter()
            for m in wm + wp:
                m.free()
            log.free()
            if best is None or t3 - t0 < best[0]:
                best = (t3 - t0, t1 - t0, t2 - t1, t3 - t2)
        tsec = torch.tensor([best[0]], dtype=torch.float64, device="cuda")
        if dist is not None:
            dist.all_reduce(tsec, op=dist.ReduceOp.MAX)
        with_witness = {"what": "program -> proof: host interpreter (serial), logs to the device, row fill + memory-log sort on the GPU, prove",
                        "rows_per_s": rows / float(tsec.item()), "s_total": float(tsec.item()), "s_host_interpreter": best[1], "s_device_witness": best[2],
                        "s_prove": best[3], "proof_equals": bool(proof_w == proof),
                        "host_row_fill_path": {"s_host_interpreter_and_row_fill": tracegen_s, "s_e2e_prove": ms_e2e / args.steps / 1e3,
                                               "rows_per_s": rows / (tracegen_s + ms_e2e / args.steps / 1e3)}}
    except Exception as exc:   # noqa: BLE001
        with_witness = {"error": "%s: %s" % (type(exc).__name__, exc)}

    # ---- N > 1, beside the headline: N independent proofs (one per GPU, no collective) — the zkVM-segment throughput ----
    replicas = None
    if dist is not None and not args.no_replicas:
        try:
            ctx.set_sharding(False)
            for m in dm + dp:
                m.free()
            dm = [ctx.upload(m) for m in traces.main]
            dp = [ctx.upload(m) for m in traces.preprocessed]
            steps_r = min(args.steps, 3)
            for _ in range(2):
                proof_r = vb.prove_machine(cfg, traces, device_resident=(dm, dp))
            barrier()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            r0.record(stream)
            for _ in range(steps_r):
                vb.prove_machine(cfg, traces, device_resident=(dm, dp))
            r1.record(stream)
            barrier()
            rep_value, rep_ms = aggregate_throughput(dist, rows * steps_r, r0.elapsed_time(r1), device="cuda", sum_rows=True)
            replicas = {"what": "%d independent proofs per step, one per GPU, no collective (weak scaling of the segment throughput)" % world,
                        "rows_per_s": rep_value, "ms_per_step": rep_ms / steps_r, "proof_equals_split_proof": bool(proof_r == proof)}
        except Exception as exc:   # noqa: BLE001
            replicas = {"error": "%s: %s" % (type(exc).__name__, exc)}

    def make_line():

        peak, peak_src = peaks()
        kstats_sorted = sorted(kstats, key=lambda k: -k[2])
        kernels = [{"kernel": k[0], "launches_per_step": k[1] / args.steps, "ms_per_step": k[2] / args.steps,
                    "algorithmic_gb_per_step": k[3] / args.steps / 1e9, "achieved_gbs": (k[3] / 1e9) / (k[2] / 1e3) if k[2] > 0 else None} for k in kstats_sorted]
        top = kstats_sorted[0]
        achieved = (top[3] / 1e9) / (top[2] / 1e3)
        keccak_top = top[0] in ("compress_layer_kernel", "leaf_hash_kernel", "fri_leaf_hash_kernel")
        roofline = {"bound": "int_alu" if keccak_top else "hbm", "kernel": top[0], "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                    "peak_source": peak_src, "share_of_step": top[2] / ms_instr, "ms_per_step_instrumented": ms_instr / args.steps}
        if keccak_top:
            roofline["bound_note"] = ("the Keccak kernels run at the INT-ALU pipe's ceiling (LOP3/SHF), not at HBM's: `frac` is the HBM fraction the contract asks for, "
                                      "`int_alu_ceiling` is the binding one (ncu: sm__inst_executed_pipe_alu 99.8 %, DRAM 0.98 x algorithmic bytes)")
        # The Keccak kernels are bound by the INT ALU pipe, not by HBM (profiles/r01_summary.md section 4: 122 LOP3 + 58 SHF per
        # round at 63 lanes/clk/SM = 4.32 G Keccak-f/s on this part, 4.30 measured stand-alone): report that ceiling beside the HBM one.
        KECCAK_PEAK_GPERM = 4.43      # what the 2^24-node layer sustains at 99.8 % of the ALU pipe (profiles/r02_compress_raw.csv)
        keccak = {}
        for name, bytes_per_perm in (("compress_layer_kernel", 96.0), ("fri_leaf_hash_kernel", 72.0)):
            kk = [k for k in kstats if k[0] == name]
            if kk and kk[0][2] > 0:
                g = kk[0][3] / bytes_per_perm / (kk[0][2] / 1e3) / 1e9     # >= 1 permutation per `bytes_per_perm` algorithmic bytes
                keccak[name] = {"achieved_gperm_s": g, "frac_of_alu_ceiling": g / KECCAK_PEAK_GPERM}
        roofline["int_alu_ceiling"] = {"unit": "G Keccak-f/s", "peak": KECCAK_PEAK_GPERM, "kernels": keccak,
                                       "note": "lower bounds: injected layers and multi-block leaves run more permutations than counted",
                                       "ncu": "profiles/r02_compress_raw.csv: sm__inst_executed_pipe_alu 99.8 % (compress_layer_kernel of this round, 2^24 nodes in 3.79 ms = 4.43 G/s); r01_keccak_big_raw.csv: 92.8 % (leaf_hash_kernel)"}
        ratio, ratio_src = ncu_traffic_ratio(top[0])
        if ratio is not None:
            # GB per launch, like `achieved`: the measured DRAM/algorithmic ratio of the committed capture applied to this
            # run's average launch (ncu cannot run inside the timed region)
            roofline["traffic"] = ratio * (top[3] / top[1]) / 1e9
            roofline["algorithmic_gb_per_launch"] = (top[3] / top[1]) / 1e9
            roofline["traffic_source"] = "%s: DRAM read+write = %.3f x algorithmic bytes" % (ratio_src, ratio)
        ntt = [k for k in kstats if k[0] == "ntt_pass_kernel"]
        if ntt:
            a = (ntt[0][3] / 1e9) / (ntt[0][2] / 1e3)
            roofline["ntt_pass"] = {"achieved": a, "frac": a / peak, "unit": "GB/s", "bytes": "8 B per element per pass (read+write)"}
            # What bounds a pass (ncu --set full of the shipping kernel, profiles/r02_ntt_v7_raw.csv + the source page): it is ISSUE bound,
            # not HBM bound.  A radix-2 butterfly on 32-bit Montgomery words is 8 instructions (3 IMAD for the product, 3 adds, 2 min) =
            # 4 per element-stage; a 14-stage pass executes 100.5 instructions per element (67 arithmetic — 56 butterfly floor + the
            # inter-pass twiddle and its running product — 13.5 shared-memory accesses, 20 addressing / control) at 57-62 % issue-slot
            # utilisation (two-way bank conflicts on the last radix-4 step, math-pipe throttle).  At the butterfly floor and full issue a
            # pass would run at about the HBM peak; a transform is two passes, so its ALGORITHMIC rate (8 B per element per transform)
            # is capped at half of whatever a pass reaches: 50 % of HBM at best, the north star's 70 % is not reachable in two passes.
            sm_hz = (clocks.get("sm_mhz") or 1965) * 1e6
            issue = 148 * 128 * sm_hz                                   # thread-instructions per second, one per lane per clock
            roofline["ntt_pass"]["ceiling"] = {
                "bound": "issue slots (INT32 butterflies), not HBM",
                "gbs_per_pass_at_butterfly_floor": 8.0 * issue / (11.5 * 4) / 1e9,      # 11.5 stages per pass on average, 4 instructions per element-stage
                "algorithmic_cap_of_a_two_pass_transform": "half of the per-pass rate",
                "measured": {"instructions_per_element_14_stage_pass": 100.5, "of_which_arithmetic": 67, "butterfly_floor": 56, "issue_active_pct": "57-62",
                             "gbs_per_pass_ncu": {"2^8-stage column pass": 3010, "2^10": "1580-2260", "2^14-stage row pass": "1460-1640"}},
                "source": "profiles/r02_ntt_v7_raw.csv (ncu --set full, shipping kernel), profiles/r02_summary.md"}

        # ---- second headline figure: BASELINE config 2 — 2^20 x 64 BabyBear NTT + inverse, device resident ----
        ntt_line = None
        if world == 1:
            hh, ww = 1 << 20, 64
            rr = np.arange(hh, dtype=np.uint64)[:, None]
            cc = np.arange(ww, dtype=np.uint64)[None, :]
            x = ((rr * 64 + cc) * 0x9E3779B1 % vb.BABYBEAR_P).astype(np.uint32)     # SURVEY 8(d) config 2 input
            dft = vb.Radix2Dft(ctx)
            dx = ctx.upload(x)
            for _ in range(3):
                dft.dft_batch(dx); dft.idft_batch(dx)
            torch.cuda.synchronize()
            n0, n1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = 10
            n0.record(stream)
            for _ in range(reps):
                dft.dft_batch(dx); dft.idft_batch(dx)
            n1.record(stream)
            torch.cuda.synchronize()
            ms_pair = n0.elapsed_time(n1) / reps
            roundtrip_ok = bool(np.array_equal(dx.download(), x))
            gbs = 2 * 8.0 * hh * ww / (ms_pair / 1e3) / 1e9      # two transforms, 8 B per element each (read once + write once)
            ntt_line = {"workload": "2^20 x 64 NTT + iNTT (natural order in/out), 256 MiB working set > L2", "ms_forward_plus_inverse": ms_pair,
                        "achieved": gbs, "unit": "GB/s", "frac": gbs / peak, "bytes": "8*h*w per transform", "roundtrip_bit_exact": roundtrip_ok}
            dx.free()
            # SURVEY 8(d) config 2 also asks for the one-column and the CPU-chip-width shapes; they are extras to the line:
            # any failure is recorded here and changes nothing above
            try:
                others = {}
                for w2 in (51, 1):
                    x2 = np.ascontiguousarray(x[:, :w2])
                    d2 = ctx.upload(x2)
                    for _ in range(3):
                        dft.dft_batch(d2); dft.idft_batch(d2)
                    torch.cuda.synchronize()
                    m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    m0.record(stream)
                    for _ in range(reps):
                        dft.dft_batch(d2); dft.idft_batch(d2)
                    m1.record(stream)
                    torch.cuda.synchronize()
                    ms2 = m0.elapsed_time(m1) / reps
                    ok2 = bool(np.array_equal(d2.download(), x2))
                    d2.free()
                    g2 = 2 * 8.0 * hh * w2 / (ms2 / 1e3) / 1e9
                    others["2^20 x %d" % w2] = {"ms_forward_plus_inverse": ms2, "achieved": g2, "unit": "GB/s", "frac": g2 / peak, "roundtrip_bit_exact": ok2,
                                               "l2": "working set %d MiB %s L2" % (hh * w2 * 4 >> 20, ">" if hh * w2 * 4 > 126 << 20 else "fits in")}
                ntt_line["other_widths"] = others
            except Exception as exc:   # noqa: BLE001
                ntt_line["other_widths"] = {"error": "%s: %s" % (type(exc).__name__, exc)}

        cpu_baseline = None
        if not args.no_cpu_baseline and world == 1:
            try:
                cpu_baseline = cpu_baseline_leg(workload, min(args.cpu_baseline_log_rows, log_rows))
            except Exception as exc:   # noqa: BLE001 — the GPU figures above must reach the line whatever happens here
                cpu_baseline = {"error": "%s: %s" % (type(exc).__name__, exc)}

        G = world
        line = {
            "metric": METRIC + (" (Fibonacci)" if workload == "fib" else " (multi-chip program)"), "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_total_max / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": DTYPE, "data": "synthetic",
            "config": {"workload": workload_name(workload, log_rows), "program": what, "trace_bytes": trace_bytes, "proof_bytes": len(proof),
                       "l2": "inputs (%.2f GB of traces, %.1f GB of LDEs) exceed L2" % (trace_bytes / 1e9, 4.5 * trace_bytes / 1e9),
                       "parallelism": ("ONE proof per step split across %d GPUs: trace columns shard for the coset LDE, one peer-store exchange over NVLink into "
                                       "contiguous row shards, sub-tree / quotient / openings / FRI per rank, %d x 32 B sub-roots all-gathered" % (G, G)) if G > 1 else "single GPU",
                       "host_tracegen_s": tracegen_s},
            "e2e": {"value": e2e_value, "unit": "rows/s", "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": len(proof) * G,
                    "note": "every rank copies its rows of the tall traces (1/N of them) and the short traces whole; every rank reads the proof back; `value` is from page-locked (torch pinned) buffers",
                    "other_host_memory": e2e_other},
            "gpu_launches": launches,
            "clocks": clocks,
            "roofline": roofline,
            "ntt": ntt_line,
            "cpu_baseline": cpu_baseline,
            "phases_ms": {p[0]: p[1] for p in phases},
            "kernels": kernels,
            "e2e_with_witness": with_witness,
        }
        if G > 1:
            per = 1.0 / args.steps
            line["split"] = {"proof_bytes_identical_across_ranks": proofs_identical,
                             "collectives_per_proof_rank0": {k: {"calls": v[0] * per, "mb_to_peers": v[1] * per / 1e6} for k, v in comm.items()},
                             "note": "exchange = kernels storing through peer pointers (rows->columns before the LDE, extended columns->row shards after it); "
                                     "allgather = sub-roots, LogUp totals, per-rank column sums, the FRI layer that stops being split, the opened rows; ms in `kernels`"}
            line["replicas"] = replicas
        return line

    if rank == 0:
        emit(make_line())
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
