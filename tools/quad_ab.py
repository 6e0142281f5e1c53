"""A/B of the 128-channel pipeline kernels: trunk_quad_kernel (4 positions per CTA, one CTA per SM; what an unforced
context with >= 4 slots launches) against trunk_duo_kernel (2 positions per CTA, two CTAs per SM; NSB_TRUNK128=duo).

Per round, alternating legs: `bench.py --config 2` (10 x 128, B = 256, 4 slots) in a subprocess, once with
NSB_TRUNK128=duo and once unforced; from each line the rate (`value`), the clocks, the board's energy per evaluation
(`roofline.energy`, from the NVML energy counter over the timed region) and the isolated launch.  Then one sweep pass
(tools/sweep.py's trunk sweep: CUDA events, 1 and 4 streams) of both kernels at B = 256 ... 4096 with 4 slots, and the
card's name and power limit read in the same run.  One JSON object on stdout and in `--out`.

    python tools/quad_ab.py [--rounds 3] [--steps 20] [--warmup 5] [--out profiles/r4_quad_ab.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))

LEGS = {"duo": "duo", "default": None}   # leg -> NSB_TRUNK128


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in out.stdout.strip().split(",")))) if out.returncode == 0 else {}


def env_for(force):
    env = dict(os.environ)
    env.pop("NSB_TRUNK128", None)
    if force:
        env["NSB_TRUNK128"] = force
    return env


def bench_leg(args, force):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", "2", "--steps", str(args.steps),
           "--warmup", str(args.warmup), "--no-selfplay", "--no-cpu-baseline"]
    out = subprocess.run(cmd, capture_output=True, text=True, env=env_for(force), cwd=ROOT)
    if out.returncode != 0:
        raise SystemExit(f"quad_ab: bench.py failed ({force}):\n{out.stdout[-2000:]}\n{out.stderr[-4000:]}")
    line = json.loads(out.stdout.strip().splitlines()[-1])
    rf = line.get("roofline", {})
    clk = line.get("clocks") or {}
    return {"value": line["value"], "kernel": rf.get("kernel"), "energy": rf.get("energy"),
            "energy_counter": clk.get("energy_counter"),
            "clocks": {k: clk.get(k) for k in ("sm_mhz", "sm_mhz_min", "sm_max_mhz", "power_w_median", "reasons") if k in clk},
            "isolated_launch": rf.get("isolated_launch")}


def sweep_pass(batches):
    import sweep   # tools/sweep.py (loads the package on import)
    rows = {}
    for leg, force in LEGS.items():
        if force:
            os.environ["NSB_TRUNK128"] = force
        else:
            os.environ.pop("NSB_TRUNK128", None)
        got = []
        sweep.trunk_sweep([(128, 10)], batches, got.append)
        rows[leg] = {r["batch"]: {k: r[k] for k in ("latency_ms", "evals_per_s_1stream", "evals_per_s_4streams")} for r in got}
    os.environ.pop("NSB_TRUNK128", None)
    return {str(b): {"duo": rows["duo"][b], "quad": rows["default"][b],
                     "ratio_4streams": round(rows["default"][b]["evals_per_s_4streams"] / rows["duo"][b]["evals_per_s_4streams"], 4)}
            for b in batches}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batches", default="256,512,1024,2048,4096")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_quad_ab.json"))
    args = ap.parse_args()
    info = {"card_before": card()}
    rounds = []
    for r in range(args.rounds):
        row = {}
        for leg in (("duo", "default") if r % 2 == 0 else ("default", "duo")):
            row[leg] = bench_leg(args, LEGS[leg])
        row["ratio"] = round(row["default"]["value"] / row["duo"]["value"], 4)
        rounds.append(row)
    vals = {leg: [r[leg]["value"] for r in rounds] for leg in LEGS}
    uj = {leg: [r[leg]["energy"]["uj_per_eval"] for r in rounds if r[leg].get("energy")] for leg in LEGS}
    summary = {leg: {"median": statistics.median(v), "min": min(v), "max": max(v),
                     "spread": round((max(v) - min(v)) / statistics.median(v), 4),
                     "uj_per_eval_median": statistics.median(uj[leg]) if uj[leg] else None} for leg, v in vals.items()}
    result = {
        "what": "bench.py --config 2 (10x128, B=256, 4 slots): unforced (trunk_quad_kernel) vs NSB_TRUNK128=duo, alternating",
        "card": info["card_before"], "card_after": card(),
        "kernels": {leg: rounds[0][leg]["kernel"] for leg in LEGS},
        "summary": summary,
        "ratio_median": round(summary["default"]["median"] / summary["duo"]["median"], 4),
        "every_default_round_above_every_duo_round": min(vals["default"]) > max(vals["duo"]),
        "rounds": rounds,
        "sweep_10x128_4slots": sweep_pass([int(b) for b in args.batches.split(",")]),
    }
    text = json.dumps(result)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")


if __name__ == "__main__":
    main()
