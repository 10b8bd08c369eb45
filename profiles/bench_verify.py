"""Proofs/s of Machine::verify: vgpu_verify one proof at a time (host checks) against vgpu_verify_batch (device checks) at batch
sizes 1, 16, 64, 256, for three workloads: Fibonacci 2^16-row proofs of several distinct n (each with its own program ROM), the
2^22-row Fibonacci proof repeated, and the config-5 program.  Every batch size is warmed up once before it is timed, and every
batch's verdicts are checked against vgpu_verify's.  Prints ONE JSON line: throughputs, per-kernel-class device times of one timed
batch (vgpu_ctx_kernel_stats), the host stretches of that batch (decode, transcripts, packing) and the GPU name and power limit,
read in the same run.

    python profiles/bench_verify.py [--sizes 1,16,64,256] [--single-reps 3] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,power.max_limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, limit, max_limit = [s.strip() for s in out.split(",")]
        return {"gpu": name, "power_limit": limit, "power_max_limit": max_limit}
    except Exception as e:   # noqa: BLE001 — the numbers still stand, without the label
        return {"gpu": "unknown (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="1,16,64,256")
    ap.add_argument("--single-reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sizes = [int(s) for s in args.sizes.split(",")]

    import oracle_binding
    import programs
    import valida_b200 as vb

    ctx = vb.Context(0)
    cfg = vb.StarkConfig(ctx, oracle_binding.Oracle().rc480)

    keep = []   # the traces objects own the memory their preprocessed arrays view

    def prove(prog):
        t = vb.run_program(prog, initial_fp=0x1000)
        keep.append(t)
        return vb.prove_machine(cfg, t), t.preprocessed

    workloads = {}
    fib16 = [prove(vb.fib_program(n)) for n in (9360, 9355, 9350, 9345)]   # 2^16-row CPU traces, four distinct ROMs
    workloads["fib_2^16_x4_programs"] = fib16
    workloads["fib_2^22"] = [prove(vb.fib_program(599183))]
    workloads["config5"] = [prove(programs.config5_program(60))]

    result = {"metric": "verified proofs/s", **gpu_info(), "host_threads_decode_transcript": 8, "workloads": {}}
    for name, items in workloads.items():
        proofs = [p for p, _ in items]
        preps = [pp for _, pp in items]
        w = {"proof_bytes": [len(p) for p in proofs]}
        # one at a time through vgpu_verify
        t0 = time.perf_counter()
        n_single = 0
        for _ in range(args.single_reps):
            for p, pp in items:
                vb.verify_machine(cfg, p, pp)
                n_single += 1
        w["vgpu_verify_proofs_per_s"] = n_single / (time.perf_counter() - t0)
        w["batch"] = {}
        for b in sizes:
            batch = [proofs[i % len(proofs)] for i in range(b)]
            prog_of = [i % len(proofs) for i in range(b)]
            got = vb.verify_machines(cfg, batch, preps, program_of=prog_of)   # warm-up
            assert got == [0] * b, got
            ctx.set_kernel_timing(True)
            ctx.kernel_stats()
            t0 = time.perf_counter()
            got = vb.verify_machines(cfg, batch, preps, program_of=prog_of)
            dt = time.perf_counter() - t0
            ks = ctx.kernel_stats()
            ctx.set_kernel_timing(False)
            assert got == [0] * b, got
            w["batch"][str(b)] = {
                "proofs_per_s": b / dt, "wall_ms": dt * 1e3,
                "kernels_ms": {k: round(ms, 4) for k, _, ms, _ in ks},
                "kernel_launches": {k: n for k, n, _, _ in ks},
                "stretches_ms": {k: round(v, 3) for k, v in vb.last_verify_batch_phases(ctx)},
            }
        best = max(w["batch"].values(), key=lambda r: r["proofs_per_s"])["proofs_per_s"]
        w["best_batch_speedup_vs_vgpu_verify"] = best / w["vgpu_verify_proofs_per_s"]
        result["workloads"][name] = w
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
