"""A/B of a 192-channel net on trunk_pair_kernel<192> against the same net zero-padded to 256 channels
(weights_io.pad_channels) on the 256-channel kernel - what running such a net costs without the 192 kernel.

Per round, alternating legs: bench.py's device-resident production step (fused decode, B positions per launch,
`--slots` streams, inputs rotating over a pool larger than L2) for at least `--seconds`; evals/s, useful TFLOP/s
(bench.trunk_flops_per_sample at the net's real width) and their share of the measured bf16 peaks.  Then the isolated
launch of each leg at B, the card's name, power limit and SM clocks, and a check that both legs return the same bits
for the same batches.  One JSON line on stdout.

    python tools/width_ab.py [--blocks 20] [--batch 512] [--slots 4] [--rounds 3] [--seconds 1.5]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import __graft_entry__ as graft  # noqa: E402
import bench  # noqa: E402

PEAK_BURST, PEAK_SUSTAINED = 1613.1, 1356.4   # bf16 dense TFLOP/s measured on this project's B200 (BASELINE.md)


def card():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "--id=0", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (x.strip() for x in out.stdout.strip().split(",")))) if out.returncode == 0 else {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=20)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--slots", type=int, default=4)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=1.5, help="least length of each timed region")
    ap.add_argument("--seed", type=int, default=1234)
    args = ap.parse_args()
    pkg = graft.load_package()
    nb, synth, rep, wio = pkg.binding, pkg.synth, pkg.replica, pkg.weights_io
    if nb.device_count() < 1:
        raise SystemExit("width_ab: no CUDA device; the product path has no CPU fallback")
    B, S = args.batch, args.slots
    desc = nb.net_desc(192, args.blocks)
    blob = nb.random_blob(desc, args.seed)
    legs = {"192": (desc, blob), "padded256": (nb.net_desc(256, args.blocks), wio.pad_channels(blob, desc, 256))}
    ctxs, wls, names = {}, {}, {}
    for k, (d, b) in legs.items():
        ctxs[k] = nb.Context(d, batch_max=B, slots=S, blob=b)
        wls[k] = bench.Workload(nb, synth, ctxs[k], B, 0)
        names[k] = ctxs[k].trunk_kernel_name()
    flops = bench.trunk_flops_per_sample(192, args.blocks)

    # batches per timed region, from a short leg of the slower kernel
    ms, _, _ = bench.device_leg(nb, rep, ctxs["padded256"], wls["padded256"], S, 64, 16)
    batches = S * math.ceil(args.seconds * 1000.0 / (ms / 64) / S)
    sampler = bench.ClockSampler(0)
    sampler.start()
    rounds = []
    for r in range(args.rounds):
        row = {}
        for k in (("192", "padded256") if r % 2 == 0 else ("padded256", "192")):
            elapsed_ms, _, (t0, t1) = bench.device_leg(nb, rep, ctxs[k], wls[k], S, batches, 8 * S)
            rate = batches * B / (elapsed_ms / 1000.0)
            clk = sampler.window(t0, t1) or {}
            row[k] = {"evals_per_s": round(rate, 1), "seconds": round(elapsed_ms / 1000.0, 3), "batches": batches,
                      "useful_tflops": round(rate * flops / 1e12, 1), "sm_mhz": clk.get("sm_mhz"),
                      "power_w_median": clk.get("power_w_median"), "reasons": clk.get("reasons")}
        row["ratio"] = round(row["192"]["evals_per_s"] / row["padded256"]["evals_per_s"], 4)
        rounds.append(row)
    sampler.stop()

    iso = {}
    for k in legs:
        launch_ms, seq_ms, n, _ = bench.isolated_leg(nb, ctxs[k], wls[k], 200)
        iso[k] = {"launch_ms": round(launch_ms, 4), "launches": n, "useful_tflops": round(B * flops / (launch_ms / 1000.0) / 1e12, 1)}

    # same inputs, same batches: the two legs must agree bit for bit at the timed size
    outs = {}
    for k in legs:
        for i in range(wls[k].n_out):
            wls[k].dev_step(ctxs[k], i, 0)
        ctxs[k].await_(0)
        outs[k] = wls[k].outputs(range(wls[k].n_out))
    identical = all(np.array_equal(outs["192"][f].view(np.uint32), outs["padded256"][f].view(np.uint32)) for f in outs["192"])
    for k in legs:
        wls[k].free()
        ctxs[k].close()

    med = {k: statistics.median(r[k]["evals_per_s"] for r in rounds) for k in legs}
    summary = {k: {"evals_per_s": round(v, 1), "useful_tflops": round(v * flops / 1e12, 1),
                   "frac_of_burst": round(v * flops / 1e12 / PEAK_BURST, 4),
                   "frac_of_sustained": round(v * flops / 1e12 / PEAK_SUSTAINED, 4)} for k, v in med.items()}
    print(json.dumps({
        "what": f"{args.blocks}x192 on trunk_pair_kernel<192> vs the same net zero-padded to 256 channels, B={B}, {S} slots",
        "card": card(), "kernels": names, "gflop_per_position_useful": round(flops / 1e9, 4),
        "peaks_tflops": {"burst": PEAK_BURST, "sustained": PEAK_SUSTAINED},
        "median": summary, "ratio_median": round(med["192"] / med["padded256"], 4), "rounds": rounds,
        "isolated_launch": iso, "isolated_ratio": round(iso["padded256"]["launch_ms"] / iso["192"]["launch_ms"], 4),
        "outputs_bit_identical": bool(identical)}))
    if not identical:
        sys.exit(1)


if __name__ == "__main__":
    main()
