"""Joules per evaluation, measured: the board's NVML energy counter around (a) the bench's timed region with the one-CTA
kernel, (b) the same with the duo kernel, (c) a back-to-back cuBLAS bf16 GEMM (torch.matmul 8192^3) for the same time.
DESIGN.md 9 argues that the steady state is energy-bound; this is the measurement behind its pJ-per-FLOP figures.

    python tools/energy_ab.py [--seconds 3] > profiles/rN_energy_ab.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bench_line(env, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "5", "--no-selfplay",
                          "--no-cpu-baseline", "--no-latency-leg"], capture_output=True, text=True, env={**os.environ, **env}, timeout=900)
    if out.returncode != 0:
        return {"error": out.stderr[-400:]}
    d = json.loads(out.stdout.strip().splitlines()[-1])
    return {"kernel": d["roofline"]["kernel"], "mode": env.get("NSB_TRUNK128"), "evals_per_s": d["value"], "clocks": d["clocks"], "energy": d["roofline"].get("energy"),
            "frac_of_burst": d["roofline"]["frac"]}


def matmul_energy(seconds):
    import pynvml
    import torch
    pynvml.nvmlInit()
    h = pynvml.nvmlDeviceGetHandleByIndex(0)
    n = 8192
    a = torch.randn(n, n, device="cuda", dtype=torch.bfloat16)
    b = torch.randn(n, n, device="cuda", dtype=torch.bfloat16)
    for _ in range(20):
        a @ b
    torch.cuda.synchronize()
    # reach the steady state first (the cap bites after a few hundred milliseconds), then count
    t_end = time.perf_counter() + 1.0
    while time.perf_counter() < t_end:
        for _ in range(20):
            a @ b
        torch.cuda.synchronize()
    e0, t0, it = pynvml.nvmlDeviceGetTotalEnergyConsumption(h), time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        for _ in range(20):
            a @ b
        torch.cuda.synchronize()
        it += 20
    t1, e1 = time.perf_counter(), pynvml.nvmlDeviceGetTotalEnergyConsumption(h)
    joules, flops = (e1 - e0) / 1000.0, 2.0 * n ** 3 * it
    return {"what": "torch.matmul bf16 8192^3 back to back", "tflops": round(flops / (t1 - t0) / 1e12, 1),
            "avg_power_w": round(joules / (t1 - t0), 1), "pj_per_flop": round(joules / flops * 1e12, 4),
            "sm_mhz_end": pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=3.0)
    args = ap.parse_args()
    steps = max(20, int(args.seconds / 0.053))
    out = {"one_cta_kernel": bench_line({"NSB_TRUNK128": "classic"}, steps), "duo_kernel": bench_line({"NSB_TRUNK128": "duo"}, steps),
           "cublas": matmul_energy(args.seconds)}
    for k in ("one_cta_kernel", "duo_kernel"):
        e = out[k].get("energy")
        if e:
            e["pj_per_executed_flop"] = round(e["pj_per_useful_flop"] * 162.0 / 192.0, 4)
    print(json.dumps(out, indent=1))


if __name__ == "__main__":
    main()
