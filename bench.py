#!/usr/bin/env python
"""bench.py — leaf evals/sec of the B200 leaf-evaluation path (BASELINE.json metric).

A STEP is a fixed bundle of `config.batches_per_step` batches (so that the timed region is about a second under the
driver's `--steps 20`, long enough for the board to reach its steady clocks and for the clock sampler to see it); a
batch is one pass of the hot path over B synthetic positions: feature bitboards -> (in-kernel plane expansion) -> ResNet
on tcgen05 -> policy head -> fused legal-move gather + softmax + value/draw sigmoids.  One kernel launch per batch.

  --config 2 (default): 10 x 128 net, B = 256        the configuration BASELINE.json's metric is quoted on
  --config 3          : 20 x 256 net, B = 512        (USI `go`: executor-side evals/s + one-batch-in-flight latency;
                                                      the search itself needs libnshogi's rules, DESIGN.md §2)
  --config 4          : 20 x 256 net, B = 512        + the self-play loop (1024 concurrent games per GPU)
  --config 5          : 40 x 256 net, B = 1024       + the batch sweep 64 .. 4096 (TFLOP/s, % of burst / sustained peak)

  value : device-timed (CUDA events on the launch streams), inputs already resident in HBM, rotating over a pool of
          input batches larger than L2, `streams_in_flight` batches in flight.
  e2e   : the same step through the host-buffer C-ABI call (nsb_eval_decode_async + nsb_await): pinned host inputs,
          H2D + kernel + D2H inside the timed region; e2e.infer_contract is the unmodified Infer contract (dense logits).
  --impl reference : the reference's CPU path for its CPU-runnable config (pack + its own Random executor, compiled into
          oracle/_ref when the reference's sources are given, else its port + decode) on all host cores.
  --dump-outputs DIR : after the timed steps, the results of the last step's final batches as DIR/<name>.npy.
Multi-GPU: one process per GPU (torchrun), independent replicas, weak scaling; NCCL only for the barrier, the
max-over-ranks of the timed region and the final counter reduction.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as graft  # noqa: E402

UNIT = "evals/s"
L2_BYTES = 126 * 1024 * 1024

# channels, blocks, batch, batches per step, weight seed (seeds with a live value head, tests/test_depth_parity.py)
CONFIGS = {
    2: dict(channels=128, blocks=10, batch=256, batches_per_step=512, seed=1,
            name="bench: 10-block 128-ch ResNet random-init, batch 256 leaf evaluation on 1xB200"),
    3: dict(channels=256, blocks=20, batch=512, batches_per_step=32, seed=1234,
            name="USI go, 20-block 256-ch ResNet, batch 512, 1xB200: executor-side leaf evals/s (search needs libnshogi)"),
    4: dict(channels=256, blocks=20, batch=512, batches_per_step=32, seed=1234,
            name="self-play data generation, 20x256 ResNet, 1024 concurrent games per GPU"),
    5: dict(channels=256, blocks=40, batch=1024, batches_per_step=8, seed=5,
            name="large-batch sweep 64-4096 on 40-block 256-ch ResNet, tensor-pipe roofline report"),
}


def metric_name(B):
    return f"nn_leaf_evals_per_sec_batch{B}"


def make_config(args):
    """The `config` object of the JSON line: identical for the b200 arm and the reference arm of one --config."""
    c = CONFIGS[args.config]
    return {"workload": f"{c['name']} (feature planes + forward + policy decode), per replica", "config": args.config,
            "batch": args.batch, "channels": args.channels, "blocks": args.blocks, "batches_per_step": args.batches_per_step,
            "launches_per_batch": 1, "streams_in_flight": args.slots,
            "l2_policy": "inputs rotate over a pool of batches larger than L2 (126 MiB); weights stay L2-resident as in "
                         "steady-state serving"}


def trunk_flops_per_sample(C, blocks, in_ch=86):
    """2*MACs, unpadded channels (SURVEY.md §8d): stem + 2*blocks convs + policy/value heads + FCs."""
    conv = lambda ci, co, k: 2.0 * 81 * k * ci * co
    f = conv(in_ch, C, 9) + 2 * blocks * conv(C, C, 9) + conv(C, 27, 1) + conv(C, 1, 1)
    f += 2.0 * 81 * 256 + 2.0 * 256 * 2
    return f


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops", 1590.0), d.get("bf16_tflops_sustained", 1400.0), d.get("hbm_gbs", 6650.0), "measured"
    return 1590.0, 1400.0, 6650.0, "fallback"


class ClockSampler:
    """SM clock, power and throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks line).  NVML in
    a thread of this process (every 20 ms, time-stamped, so that the samples inside a window can be picked out exactly);
    falls back to `nvidia-smi -lms 100` when NVML cannot be loaded."""

    SMI_Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []          # (t, sm_mhz, power_w, reasons bitmask)
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._smi = None
        self._smi_lines = []
        self.source = None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = self.gpu
            if vis:
                ids = [v.strip() for v in vis.split(",") if v.strip()]
                if self.gpu < len(ids) and ids[self.gpu].isdigit():
                    phys = int(ids[self.gpu])
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            reasons_fn = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons

            def loop():
                while not self._stop.is_set():
                    try:
                        try:
                            mj = float(pynvml.nvmlDeviceGetTotalEnergyConsumption(h))   # the board's own energy counter, mJ
                        except pynvml.NVMLError:
                            mj = None
                        self.samples.append((time.perf_counter(), float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)),
                                             pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0, int(reasons_fn(h)), mj))
                    except pynvml.NVMLError:
                        pass
                    self._stop.wait(0.02)

            self._thread = threading.Thread(target=loop, daemon=True)
            self._thread.start()
            self.source = "nvml, 20 ms"
        except Exception:  # noqa: BLE001 - any NVML problem: use the command-line tool
            try:
                self._smi = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.SMI_Q}",
                                              "--format=csv,noheader,nounits", "-lms", "100"],
                                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
                threading.Thread(target=self._pump, daemon=True).start()
                self.source = "nvidia-smi -lms 100"
            except OSError:
                self._smi = None

    def _pump(self):
        for line in self._smi.stdout:
            self._smi_lines.append((time.perf_counter(), line.strip()))

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)
        if self._smi is not None:
            self._smi.terminate()
            try:
                self._smi.wait(timeout=5)
            except subprocess.TimeoutExpired:
                self._smi.kill()
            for t, ln in self._smi_lines:
                f = [x.strip() for x in ln.split(",")]
                if len(f) < 9:
                    continue
                try:
                    mask = 0
                    for bit, v in zip((0x8, 0x40, 0x20, 0x4), f[5:9]):   # NVML's bit values for the same four reasons
                        if v.lower().startswith("active"):
                            mask |= bit
                    self.samples.append((t, float(f[1]), float(f[3]), mask))
                    self.max_mhz = float(f[2])
                except ValueError:
                    continue

    def window(self, t0: float, t1: float):
        """Summary of the samples taken in [t0, t1] (perf_counter times)."""
        inside = [s for s in self.samples if t0 <= s[0] <= t1]
        if not inside:
            return None
        names = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}
        reasons = sorted({nm for s in inside for bit, nm in names.items() if s[3] & bit})
        out = {"sm_mhz": statistics.median(s[1] for s in inside), "sm_mhz_min": min(s[1] for s in inside),
               "sm_max_mhz": self.max_mhz, "power_w_max": round(max(s[2] for s in inside), 1),
               "power_w_median": round(statistics.median(s[2] for s in inside), 1), "samples": len(inside),
               "reasons": reasons, "window_s": round(t1 - t0, 3), "source": self.source,
               "window": "the timed region of `value` only"}
        # energy from the board's counter between the first and the last sample inside the window (the counter's own
        # average power over that span; the instantaneous power readings above lag by NVML's averaging window)
        counted = [s for s in inside if len(s) > 4 and s[4] is not None]
        if len(counted) >= 2 and counted[-1][0] > counted[0][0]:
            joules = (counted[-1][4] - counted[0][4]) / 1000.0
            out["energy_counter"] = {"joules": round(joules, 2), "span_s": round(counted[-1][0] - counted[0][0], 3),
                                     "avg_power_w": round(joules / (counted[-1][0] - counted[0][0]), 1)}
        return out


class Workload:
    """Synthetic inputs of one (net, batch): a device pool of feature-bitboard batches larger than L2 (built with the
    product's own stage-1 kernel from packed synthetic positions), CSR legal-move lists, output buffers."""

    def __init__(self, nb, synth, ctx, B, rank, small_pool=False):
        self.nb, self.B = nb, B
        self.fb_bytes = B * 86 * 16
        self.pool = max(4, (L2_BYTES + self.fb_bytes - 1) // self.fb_bytes + 8) if not small_pool else 8
        self.pos = synth.random_positions(2048, seed=20240203 + rank)
        d_pos = nb.DeviceBuffer.from_host(self.pos)
        d_fb_unique = nb.DeviceBuffer(len(self.pos) * 86 * 16)
        ctx.pack_positions_device(0, d_pos.ptr, len(self.pos), d_fb_unique.ptr)   # product stage-1 kernel
        ctx.await_(0)
        fb_unique = d_fb_unique.to_host((len(self.pos), 86), nb.FEATURE_BITBOARD)
        d_pos.free()
        d_fb_unique.free()
        self.rng = np.random.default_rng(99 + rank)
        self.off, self.idx = synth.random_legal_moves(B, seed=20240203, edge_rows=False)
        self.n_moves = int(self.off[-1])
        self.host_pool = fb_unique[self.rng.integers(0, len(self.pos), size=self.pool * B)].reshape(self.pool, B * 86)
        self.d_pool = nb.DeviceBuffer.from_host(self.host_pool)
        self.d_off = nb.DeviceBuffer.from_host(self.off)
        self.d_idx = nb.DeviceBuffer.from_host(self.idx)
        self.n_out = 8
        self.d_legal = [nb.DeviceBuffer(max(self.n_moves, 1) * 4) for _ in range(self.n_out)]
        self.d_win = [nb.DeviceBuffer(B * 4) for _ in range(self.n_out)]
        self.d_draw = [nb.DeviceBuffer(B * 4) for _ in range(self.n_out)]
        self.d_flag = [nb.DeviceBuffer(B) for _ in range(self.n_out)]

    def dev_step(self, ctx, i, slot=0):
        j = i % self.n_out
        # the production path: legal-move rows out, dense logits never leave the SM (d_policy = NULL)
        ctx.eval_decode_device(slot, self.d_pool.ptr + (i % self.pool) * self.fb_bytes, self.B, self.d_off.ptr, self.d_idx.ptr,
                               self.nb.DECODE_PROBS, None, self.d_legal[j].ptr, self.d_win[j].ptr, self.d_draw[j].ptr,
                               self.d_flag[j].ptr)

    def outputs(self, batches):
        """What dev_step handed back for the given batch indices, in that order: legal-move probabilities (CSR rows of
        self.off), win and draw rates, NaN flags.  A batch's buffers hold its result until batch i + n_out is launched."""
        rows = [(self.d_legal[i % self.n_out].to_host((self.n_moves,), np.float32),
                 self.d_win[i % self.n_out].to_host((self.B,), np.float32),
                 self.d_draw[i % self.n_out].to_host((self.B,), np.float32),
                 self.d_flag[i % self.n_out].to_host((self.B,), np.uint8).astype(np.float32)) for i in batches]
        return {name: np.stack(col) for name, col in zip(("legal_probs", "win", "draw", "nan_flag"), zip(*rows))}

    def free(self):
        for b in [self.d_pool, self.d_off, self.d_idx] + self.d_legal + self.d_win + self.d_draw + self.d_flag:
            b.free()


def device_leg(nb, rep, ctx, wl, slots, batches, warm_batches, step_batches=None):
    """`batches` launches round-robin over `slots` streams, device-resident inputs / outputs, CUDA events on the streams.
    Returns (elapsed ms, per-step ms list or None, perf_counter window)."""
    S = slots
    assert wl.n_out % S == 0           # an output buffer is only ever reused on the stream that wrote it last
    for i in range(warm_batches):
        wl.dev_step(ctx, i, i % S)
    for s_ in range(S):
        ctx.await_(s_)
    rep.barrier()
    nb.device_sync()
    e0 = nb.Event()
    marks = []                          # per step boundary: one event per stream
    t0 = time.perf_counter()
    e0.record(ctx, 0)
    for i in range(batches):
        wl.dev_step(ctx, warm_batches + i, i % S)
        if step_batches and (i + 1) % step_batches == 0:
            evs = [nb.Event() for _ in range(S)]
            for s_ in range(S):
                evs[s_].record(ctx, s_)
            marks.append(evs)
    if not marks or batches % (step_batches or batches):
        evs = [nb.Event() for _ in range(S)]
        for s_ in range(S):
            evs[s_].record(ctx, s_)
        marks.append(evs)
    for e in marks[-1]:
        e.sync()
    for s_ in range(S):
        ctx.await_(s_)
    nb.device_sync()
    t1 = time.perf_counter()
    rep.barrier()
    ends = [max(e0.elapsed_ms(e) for e in evs) for evs in marks]
    per_step = [b - a for a, b in zip([0.0] + ends[:-1], ends)] if step_batches else None
    for evs in marks:
        for e in evs:
            e.destroy()
    e0.destroy()
    return ends[-1], per_step, (t0, t1)


def isolated_leg(nb, ctx, wl, launches, warm=20):
    """The trunk kernel launched alone: back to back on ONE stream (no overlap between launches), one CUDA event pair
    around each launch, harvested in nsb_await.  Returns (avg launch ms, ms per step of that sub-run, launches)."""
    for i in range(warm):
        wl.dev_step(ctx, i, 0)
    ctx.await_(0)
    ctx.set_timing(True)
    ctx.trunk_time_reset()
    es0, es1 = nb.Event(), nb.Event()
    es0.record(ctx, 0)
    for i in range(launches):
        wl.dev_step(ctx, warm + i, 0)
    es1.record(ctx, 0)
    es1.sync()
    ctx.await_(0)
    seq_ms = es0.elapsed_ms(es1)
    ms_sum, n = ctx.trunk_time()
    ctx.set_timing(False)
    return ms_sum / max(n, 1), seq_ms / max(launches, 1), n, ms_sum / seq_ms if seq_ms > 0 else None


def run_b200(args):
    pkg = graft.load_package()
    nb, synth, rep = pkg.binding, pkg.synth, pkg.replica
    info = rep.RankInfo.from_env()
    world = info.world
    dev_device = None
    if world > 1 or args.gpus > 1:
        import torch
        import torch.distributed as dist

        if world != args.gpus:
            raise SystemExit(f"--gpus {args.gpus} needs torchrun with {args.gpus} ranks (WORLD_SIZE={world})")
        torch.cuda.set_device(info.local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", info.local_rank))
        dev_device = torch.device("cuda", info.local_rank)
    if nb.device_count() < 1:
        raise SystemExit("bench: no CUDA device; the product path has no CPU fallback")
    gpu = info.local_rank
    numa_bound = nb.numa_bind_thread(gpu)     # host buffers and this thread on the GPU's own NUMA node (evaluator.cc:39-83,127-136)
    B, C, blocks, slots, bps = args.batch, args.channels, args.blocks, args.slots, args.batches_per_step
    desc = nb.net_desc(C, blocks)
    blob = nb.random_blob(desc, args.seed)
    ctx = nb.Context(desc, batch_max=B, slots=slots, gpu=gpu, blob=blob)
    wl = Workload(nb, synth, ctx, B, info.rank, args.small_pool)
    K, W = args.steps, max(args.warmup, 3)
    tf_burst, tf_sust, hbm, which = peaks()
    flops_batch = trunk_flops_per_sample(C, blocks) * B

    # ---- value: K steps of `bps` batches, device-resident, `slots` streams ------------------------------------------
    sampler = ClockSampler(gpu)
    sampler.start()
    l0 = ctx.launch_count()
    elapsed_ms, per_step, (tw0, tw1) = device_leg(nb, rep, ctx, wl, slots, K * bps, W * bps, step_batches=bps)
    launches = ctx.launch_count() - l0 - W * bps
    clocks = sampler.window(tw0, tw1)
    # the results of the last step's final batches (at most 64 MiB), taken before the legs below reuse the output buffers
    end = (W + K) * bps
    n_dump = max(1, min(wl.n_out, bps, (64 << 20) // (wl.n_moves * 4 + B * 12)))
    dumped = wl.outputs(range(end - n_dump, end)) if args.dump_outputs and info.rank == 0 else None
    counters, elapsed_max = rep.aggregate({"evals": B * K * bps, "batches": K * bps, "legal_moves": wl.n_moves * K * bps},
                                          elapsed_ms, device=dev_device)
    value = rep.whole_job_rate(counters["evals"], elapsed_max)
    batch_ms = elapsed_max / (K * bps)
    achieved_ss = flops_batch / (batch_ms * 1e-3) / 1e12
    # burst (first step after the warm-up's idle gap) against steady state (second half of the run), this rank
    steady = per_step[len(per_step) // 2:] if per_step and len(per_step) >= 4 else per_step
    ss_batch_ms = (sum(steady) / len(steady) / bps) if steady else batch_ms
    best_step_ms = min(per_step) if per_step else elapsed_ms / K

    # ---- the kernel alone -------------------------------------------------------------------------------------------
    iso_n = min(max(K * bps // 4, 100), 1000)
    iso_ms, iso_step_ms, iso_launches, iso_share = isolated_leg(nb, ctx, wl, iso_n)
    isolated = {"kernel": ctx.trunk_kernel_name(), "avg_launch_ms": round(iso_ms, 5),
                "achieved": round(flops_batch / (iso_ms * 1e-3) / 1e12, 2),
                "frac": round(flops_batch / (iso_ms * 1e-3) / 1e12 / tf_burst, 4),
                "frac_of_sustained_peak": round(flops_batch / (iso_ms * 1e-3) / 1e12 / tf_sust, 4),
                "kernel_share_of_step": round(iso_share, 4) if iso_share else None,
                "timing": f"{iso_launches} launches back to back on one stream, one CUDA event pair per launch; "
                          f"that sub-run: {iso_step_ms:.5f} ms per batch"}
    one_slot = None
    if C == 128 and not args.no_latency_leg:
        # what a ONE-slot executor (the reference's usage: one batch per evaluator thread) launches for this batch size
        ctx1 = nb.Context(desc, batch_max=B, slots=1, gpu=gpu, blob=blob)
        ms1, step1, n1, share1 = isolated_leg(nb, ctx1, wl, iso_n)
        one_slot = {"kernel": ctx1.trunk_kernel_name(), "avg_launch_ms": round(ms1, 5),
                    "achieved": round(flops_batch / (ms1 * 1e-3) / 1e12, 2),
                    "frac": round(flops_batch / (ms1 * 1e-3) / 1e12 / tf_burst, 4),
                    "frac_of_sustained_peak": round(flops_batch / (ms1 * 1e-3) / 1e12 / tf_sust, 4)}
        ctx1.close()

    # ---- e2e: host buffers through the C ABI, `slots` batches in flight ----------------------------------------------
    h_pool_n = 16
    n_moves, fb_bytes = wl.n_moves, wl.fb_bytes
    h_fb = [nb.PinnedArray((B * 86,), nb.FEATURE_BITBOARD, gpu=gpu) for _ in range(h_pool_n)]
    for k, a in enumerate(h_fb):
        a.array[:] = wl.host_pool[k % wl.pool]
    h_off = nb.PinnedArray((B + 1,), np.uint32, gpu=gpu); h_off.array[:] = wl.off
    h_idx = nb.PinnedArray((max(n_moves, 1),), np.uint16, gpu=gpu); h_idx.array[:n_moves] = wl.idx
    h_legal = [nb.PinnedArray((max(n_moves, 1),), np.float32, gpu=gpu) for _ in range(slots)]
    h_win = [nb.PinnedArray((B,), np.float32, gpu=gpu) for _ in range(slots)]
    h_draw = [nb.PinnedArray((B,), np.float32, gpu=gpu) for _ in range(slots)]
    h_flag = [nb.PinnedArray((B,), np.uint8, gpu=gpu) for _ in range(slots)]
    h_policy = [nb.PinnedArray((B * 2187,), np.float32, gpu=gpu) for _ in range(slots)]
    h_pos = [nb.PinnedArray((B,), nb.POSITION, gpu=gpu) for _ in range(h_pool_n)]
    for a_ in h_pos:
        a_.array[:] = wl.pos[wl.rng.integers(0, len(wl.pos), size=B)]
    sink = 0.0

    def e2e_loop(batches, kind):
        nonlocal sink
        for i in range(batches):
            s = i % slots
            if i >= slots:
                ctx.await_(s)
                sink += float(h_win[s].array[0])            # consume the batch's result on the host
            if kind == "fused":
                ctx.eval_decode_async(s, h_fb[i % h_pool_n].array, B, h_off.array, h_idx.array, nb.DECODE_PROBS,
                                      h_legal[s].array, h_win[s].array, h_draw[s].array, h_flag[s].array)
            elif kind == "infer":
                ctx.eval_async(s, h_fb[i % h_pool_n].array, B, h_policy[s].array, h_win[s].array, h_draw[s].array)
            else:   # packed positions in: stage 1 in the trunk kernel's prologue (SURVEY.md §8 f2)
                ctx.eval_positions_decode_async(s, h_pos[i % h_pool_n].array, B, h_off.array, h_idx.array, nb.DECODE_PROBS,
                                                h_legal[s].array, h_win[s].array, h_draw[s].array, h_flag[s].array)
        for s in range(min(slots, batches)):
            ctx.await_(s)
            sink += float(h_win[s].array[0])

    def time_e2e(kind, batches):
        e2e_loop(max(bps // 4, slots), kind)
        rep.barrier()
        nb.device_sync()
        t0 = time.perf_counter()
        e2e_loop(batches, kind)
        nb.device_sync()
        dt = (time.perf_counter() - t0) * 1e3
        rep.barrier()
        _, dt_max = rep.aggregate({}, dt, device=dev_device)
        return rep.whole_job_rate(B * batches * world, dt_max)

    e2e_fused = time_e2e("fused", K * bps)
    e2e_infer = time_e2e("infer", K * bps)
    e2e_positions = time_e2e("positions", K * bps)

    # one batch at a time (the reference executor's usage: computeNonBlocking -> await per evaluator thread,
    # src/mcts/evaluationworker.cc:158-180): a one-slot context = direct I/O (the kernel reads / writes the
    # page-locked host buffers itself), against the same context with staged copies
    latency = None
    if not args.no_latency_leg:
        ctx1 = nb.Context(desc, batch_max=B, slots=1, gpu=gpu, blob=blob)
        KL = min(K * bps, 500)

        def one_at_a_time(n_batches):
            nonlocal sink
            t0 = time.perf_counter()
            for i in range(n_batches):
                ctx1.eval_decode_async(0, h_fb[i % h_pool_n].array, B, h_off.array, h_idx.array, nb.DECODE_PROBS,
                                       h_legal[0].array, h_win[0].array, h_draw[0].array, h_flag[0].array)
                ctx1.await_(0)
                sink += float(h_win[0].array[0])
            return (time.perf_counter() - t0) * 1e6 / n_batches

        latency = {"kernel": ctx1.trunk_kernel_name(), "batch": B, "batches": KL,
                   "api": "nsb_eval_decode_async + nsb_await, one batch in flight, host buffers"}
        for mode in ("staged", "direct"):
            ctx1.set_io_mode(mode == "direct")
            one_at_a_time(50)
            latency[f"{mode}_us_per_batch"] = round(one_at_a_time(KL), 2)
        latency["default_io"] = "direct"
        latency["evals_per_s_one_in_flight"] = round(B / (latency["direct_us_per_batch"] * 1e-6), 1)
        ctx1.close()
    sampler.stop()

    sweep = batch_sweep(args, nb, synth, rep, desc, blob, gpu, info, tf_burst, tf_sust) if args.config == 5 and not args.no_sweep else None
    selfplay = selfplay_leg(args, info, rep, dev_device) if args.config in (2, 4) and not args.no_selfplay else None

    # ---- roofline of the dominant (only) kernel ----------------------------------------------------------
    traffic = None
    tp = os.path.join(ROOT, "profiles", "trunk_traffic.json")
    if os.path.exists(tp):
        tag = ":duo" if "duo" in ctx.trunk_kernel_name() else ""
        traffic = json.load(open(tp)).get(f"{C}x{blocks}@{B}{tag}")
    # `achieved`: the timed region itself.  Its launches overlap (`slots` streams, CTAs of different launches share
    # the SMs), so the duration of a launch there is the steady-state time per launch, elapsed / launches; the same
    # kernel launched alone is reported beside it (isolated_launch), and so is the kernel a one-slot executor runs.
    roofline = {"bound": "tensor", "kernel": ctx.trunk_kernel_name(), "achieved": round(achieved_ss, 2),
                "peak": tf_burst, "unit": "TFLOP/s", "frac": round(achieved_ss / tf_burst, 4),
                "frac_of_sustained_peak": round(achieved_ss / tf_sust, 4), "peak_source": which,
                "peak_sustained": tf_sust,
                "peak_note": "frac is against the BURST bf16 peak of MEASURED_PEAKS.json (conservative); this kernel is timed inside a "
                             "~1 s step, for which the sustained figure is the applicable denominator: frac_of_sustained_peak",
                "flops_per_launch": flops_batch, "avg_launch_ms": round(batch_ms, 5),
                "timing": f"timed region: {K * bps} launches over {slots} streams, CUDA events on the streams, "
                          "duration per launch = elapsed / launches (launches overlap); per GPU",
                "steady_state": {"avg_launch_ms": round(ss_batch_ms, 5),
                                 "frac": round(flops_batch / (ss_batch_ms * 1e-3) / 1e12 / tf_burst, 4),
                                 "what": "second half of the timed steps (this rank): the board has reached its power-capped clock"},
                "best_step": {"avg_launch_ms": round(best_step_ms / bps, 5),
                              "frac": round(flops_batch / (best_step_ms / bps * 1e-3) / 1e12 / tf_burst, 4)},
                "isolated_launch": isolated, "one_slot_executor_launch": one_slot, "traffic": traffic}
    if clocks and clocks.get("energy_counter"):
        # joules are what the steady state is bounded by (DESIGN.md 9): the board's energy counter over the timed region
        # of this rank, per evaluation and per FLOP (useful FLOPs: the net's; the kernels execute 192 / 162 of them)
        watts = clocks["energy_counter"]["avg_power_w"]
        rate = B / (batch_ms * 1e-3)
        roofline["energy"] = {"avg_power_w": watts, "uj_per_eval": round(watts / rate * 1e6, 1),
                              "pj_per_useful_flop": round(watts / (achieved_ss * 1e12) * 1e12, 4),
                              "source": "nvmlDeviceGetTotalEnergyConsumption over the timed region, rank 0's GPU"}
    if sweep is not None:
        roofline["sweep"] = sweep

    line = {
        "metric": metric_name(B), "value": round(value, 1), "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": round(elapsed_max / K, 5), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": make_config(args),
        "e2e": {"value": round(e2e_fused, 1), "unit": UNIT, "api": "nsb_eval_decode_async + nsb_await (host buffers)",
                "h2d_bytes_per_step": (fb_bytes + (B + 1) * 4 + n_moves * 2) * bps,
                "d2h_bytes_per_step": (n_moves * 4 + B * 4 * 2 + B) * bps, "clock": "host, device-synchronised both sides",
                "infer_contract": {"value": round(e2e_infer, 1), "unit": UNIT,
                                   "api": "nsb_eval_async + nsb_await == Infer::computeNonBlocking/await (dense logits)",
                                   "h2d_bytes_per_step": fb_bytes * bps, "d2h_bytes_per_step": (B * 2187 * 4 + B * 8) * bps,
                                   "d2h_gbs_per_gpu": round(e2e_infer / world * (2187 * 4 + 8) / 1e9, 2)},
                "positions_in": {"value": round(e2e_positions, 1), "unit": UNIT,
                                 "api": "nsb_eval_positions_decode_async + nsb_await (packed positions in, stage 1 in the trunk prologue)",
                                 "h2d_bytes_per_step": (B * 108 + (B + 1) * 4 + n_moves * 2) * bps,
                                 "d2h_bytes_per_step": (n_moves * 4 + B * 4 * 2 + B) * bps},
                "one_batch_in_flight": latency,
                "host_buffers": {"numa_node_of_gpu": nb.gpu_numa_node(gpu), "thread_bound_to_node": bool(numa_bound),
                                 "alloc": "nsb_host_alloc_near (page-locked, on the GPU's NUMA node)"}},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
        "per_step_ms": [round(x, 3) for x in per_step] if per_step and len(per_step) <= 64 else None,
        "counters": counters,
    }
    if args.config == 3 and world == 1 and not args.no_selfplay:
        line["usi_go"] = usi_leg(args, info)   # measured nodes/s of a real search from the start position
    if selfplay is not None:
        line["selfplay"] = selfplay
    if info.rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(synth, B, seconds=args.cpu_seconds)
    if dumped is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, f"{name}.npy"), a)
    if info.rank == 0:
        print(json.dumps(line), flush=True)
    wl.free()
    ctx.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()
    return sink


def batch_sweep(args, nb, synth, rep, desc, blob, gpu, info, tf_burst, tf_sust):
    """BASELINE configs[4]: B = 64 .. 4096 on the 40 x 256 net: evals/s, TFLOP/s and % of burst / sustained peak per B,
    `slots` streams in flight and one launch alone."""
    rows = []
    for Bs in (64, 128, 256, 512, 1024, 2048, 4096):
        ctx = nb.Context(desc, batch_max=Bs, slots=args.slots, gpu=gpu, blob=blob)
        wl = Workload(nb, synth, ctx, Bs, info.rank, small_pool=False)
        flops = trunk_flops_per_sample(args.channels, args.blocks) * Bs
        est_ms = flops / (0.75 * tf_burst * 1e9)
        n = int(min(max(600.0 / est_ms, 8), 4000))           # ~0.6 s per point
        ms, _, _ = device_leg(nb, rep, ctx, wl, args.slots, n, max(n // 8, args.slots))
        iso_ms, _, _, _ = isolated_leg(nb, ctx, wl, max(n // 4, 4), warm=4)
        tf = flops * n / (ms * 1e-3) / 1e12
        rows.append({"batch": Bs, "launches": n, "evals_per_s": round(Bs * n / (ms * 1e-3), 1), "tflops": round(tf, 1),
                     "frac_burst": round(tf / tf_burst, 4), "frac_sustained": round(tf / tf_sust, 4),
                     "alone_launch_ms": round(iso_ms, 4), "alone_frac_burst": round(flops / (iso_ms * 1e-3) / 1e12 / tf_burst, 4)})
        wl.free()
        ctx.close()
    return rows


def selfplay_leg(args, info, rep, device):
    """BASELINE.json's second metric, "self-play positions/sec" (configs[3]: 20x256 net, 1024 concurrent
    games per GPU): the C++ self-play loop of nshogi-engine_b200/host/selfplay_real.cc (frame pool, search
    workers running a PUCT search on real shogi rules - host/rules/shogi.h, perft-pinned -, pinned multi-slot
    evaluation worker) against infer::B200, one process per GPU, counters summed over ranks."""
    exe = os.path.join(ROOT, "nshogi-engine_b200", "host", "nsb_selfplay_real")
    if not os.path.exists(exe):
        return {"unavailable": "nsb_selfplay_real not built"}
    # threads per rank: W search workers + the evaluation worker (the save worker and the main thread sleep almost always)
    workers = max(2, min(14, (os.cpu_count() or 4) // max(1, info.world) - 1))
    cmd = [exe, "--gpu", str(info.local_rank), "--channels", "256", "--blocks", "20", "--batch-size", "256", "--slots", "4",
           "--frame-pool-size", "1024", "--num-search-workers", str(workers), "--seconds", str(args.selfplay_seconds),
           "--warmup", "1.5"]
    def one_run(extra):
        rep.barrier()
        rec, err = None, None
        try:
            out = subprocess.run(cmd + extra, capture_output=True, text=True, timeout=120 + args.selfplay_seconds)
            if out.returncode == 0:
                rec = json.loads(out.stdout.strip().splitlines()[-1])
            else:
                err = out.stderr.strip()[-300:] or f"exit code {out.returncode}"
        except (OSError, subprocess.SubprocessError, ValueError, IndexError) as e:
            err = repr(e)
        # every rank takes part in the reduction, also one whose harness failed (it contributes zeros)
        mine = {"records": rec["records"], "games": rec["games"], "evals": rec["evals"], "batches": rec["batches"],
                "nan_rows": 0 if rec else 1} if rec else {"nan_rows": 1}
        counters, ms_max = rep.aggregate(mine, rec["seconds"] * 1e3 if rec else 0.0, device=device)
        if counters["nan_rows"] or rec is None:      # "nan_rows" doubles as the count of failed ranks in this reduction
            return None, {"unavailable": f"self-play harness failed on {counters['nan_rows']} rank(s): {err}"}
        return rec, {"metric": "selfplay_positions_per_sec", "value": round(rep.whole_job_rate(counters["records"], ms_max), 1),
                     "unit": "positions/s", "leaf_evals_per_sec": round(rep.whole_job_rate(counters["evals"], ms_max), 1),
                     "games_per_sec": round(rep.whole_job_rate(counters["games"], ms_max), 2),
                     "avg_batch": round(counters["evals"] / max(counters["batches"], 1), 1), "seconds": rec["seconds"]}

    rec, line = one_run([])
    if rec is None:
        return line
    line["teacher_rank0"] = rec.get("teacher")
    line["config"] = {"workload": "self-play data generation, 20x256 ResNet, 1024 concurrent games per GPU",
                      "batch_size": rec["batch_size"], "num_playouts": rec["num_playouts"], "full_search_ratio": rec["full_search_ratio"],
                      "search_workers_per_gpu": workers, "slots": rec["slots"], "rules": rec["rules"],
                      "decode": rec.get("decode"), "avg_legal_moves": rec.get("avg_legal_moves"),
                      "terminal_leaves_per_eval": rec.get("terminal_leaves_per_eval"), "eval_cache": "off: every leaf runs the network"}
    # the reference's self-play runs with an evaluation cache, 1,024 MB by default (src/selfplay/main.cc:39-40,93-106):
    # here the device-resident cache (probe kernel + store in the decode tail, DESIGN.md 6.4) of the same size
    rec_c, line_c = one_run(["--cache-mb", "1024"])
    if rec_c is not None:
        line_c["cache_mb"] = 1024
        line_c["cache_hit_rate_rank0"] = rec_c.get("cache_hit_rate")
        line_c["what"] = ("same run with the reference's default evaluation cache size (device-resident); transpositions among the "
                          "1,024 games of one random-init net are served by the probe kernel instead of the network")
    line["with_eval_cache_1GiB"] = line_c
    return line


def usi_leg(args, info):
    """BASELINE configs[2], "USI go from hirate startpos, 20-block 256-ch ResNet, batch 512, 1xB200 nodes/sec": one
    search tree from the start position (host/usi_go_bench.cc: real rules, PUCT with virtual loss, search threads
    filling the pinned batch in place, fused MCTS decode with rank order).  nps as src/protocol/usilogger.cc:46."""
    exe = os.path.join(ROOT, "nshogi-engine_b200", "host", "nsb_usi_go_bench")
    if not os.path.exists(exe) or info.rank != 0:
        return None
    threads = max(1, min(8, (os.cpu_count() or 4) - 2))
    out = {}
    for name, extra in (("search_threads_2_reference_default", ["--num-search-threads", "2"]),
                        (f"search_threads_{threads}", ["--num-search-threads", str(threads)]),
                        ("search_threads_2_device_cache_4GiB", ["--num-search-threads", "2", "--cache-mb", "4096"]),
                        (f"search_threads_{threads}_device_cache_4GiB", ["--num-search-threads", str(threads), "--cache-mb", "4096"])):
        try:
            r = subprocess.run([exe, "--gpu", str(info.local_rank), "--channels", str(args.channels), "--blocks", str(args.blocks),
                                "--batch-size", str(args.batch), "--seconds", "4"] + extra, capture_output=True, text=True, timeout=120)
            out[name] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 else {"unavailable": r.stderr.strip()[-200:]}
        except (OSError, subprocess.SubprocessError, ValueError, IndexError) as e:
            out[name] = {"unavailable": repr(e)}
    return out


def cpu_path_rate(orc, synth, B, threads, seconds):
    pos = synth.random_positions(1024, seed=20240203)
    off, idx = synth.random_legal_moves(len(pos), seed=20240203, edge_rows=False)
    use_ref = orc.have_ref_random()
    v, sec = orc.cpu_path(pos, off, idx, B, threads, 2, False, use_ref)       # calibrate
    per_thread = max(2, int(seconds / max(sec / 2, 1e-6)))
    v, sec = orc.cpu_path(pos, off, idx, B, threads, per_thread, False, use_ref)
    return v, sec, per_thread, use_ref


def cpu_baseline(synth, B, seconds=12.0):
    """The reference's CPU path for its CPU-runnable config (BASELINE.json configs[0]): stage-1 pack (port; libnshogi
    absent) + Random executor (the reference's own random.cc compiled into oracle/_ref when present, else the port) +
    decode (port), one batch per thread-iteration.  Reported twice: on every host core at this run's batch size (the
    headline `value`), and exactly as configs[0] states it - 8 threads, batch 128."""
    orc = graft.load_oracle()
    cores = os.cpu_count() or 1
    v, sec, per_thread, use_ref = cpu_path_rate(orc, synth, B, cores, seconds * 0.6)
    v0, sec0, per0, _ = cpu_path_rate(orc, synth, 128, 8, seconds * 0.4)
    # context: the same net's fp32 forward on the host cores (oracle port, vectorised C, all threads)
    pkg = graft.load_package()
    desc = pkg.binding.net_desc(128, 10)
    blob = pkg.binding.random_blob(desc, 1)
    pos = synth.random_positions(256, seed=20240203)
    planes = orc.expand(orc.pack(pos), 256)
    t0 = time.perf_counter()
    orc.forward(desc, blob, planes, False)
    fwd = 256 / (time.perf_counter() - t0)
    rand = "reference src/infer/random.cc compiled in place" if use_ref else "port of random.cc"
    return {"value": round(v, 1), "unit": UNIT, "cores": cores, "kind": "port",
            "kind_detail": f"Random executor: {rand}; stage-1 pack and decode: ports (libnshogi absent)",
            "sample": f"{cores} threads x {per_thread} batches of {B}: pack (port of FeatureStackComptime, builder-defined) + "
                      f"Random executor ({rand}) + decode (port of feedworker.cc:100-136); {sec:.1f} s; NN forward NOT "
                      "included (the reference's CPU config replaces it with the Random executor)",
            "configs0_8_threads_batch128": {"value": round(v0, 1), "unit": UNIT, "cores": 8,
                                            "sample": f"8 threads x {per0} batches of 128, same three stages; {sec0:.1f} s"},
            "with_oracle_forward_10x128": {"value": round(fwd, 1), "unit": UNIT,
                                           "sample": "256 positions through the oracle's fp32 CPU forward of the 10x128 net, all threads"}}


def run_reference(args):
    """--impl reference: the reference's CPU path on the host cores (see cpu_baseline), every core, same config object."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    pkg = graft.load_package()
    synth = pkg.synth
    orc = graft.load_oracle()
    B = args.batch
    threads = os.cpu_count() or 1
    pos = synth.random_positions(1024, seed=20240203)
    off, idx = synth.random_legal_moves(len(pos), seed=20240203, edge_rows=False)
    use_ref = orc.have_ref_random()
    v, sec = orc.cpu_path(pos, off, idx, B, threads, 2, False, use_ref)
    K, W = args.steps, max(args.warmup, 1)
    budget = 120.0                                   # whole run bounded to ~2 minutes
    per_step = max(1, int((budget / (K + W)) / max(sec / 2, 1e-6)))
    per_step = min(per_step, 64)
    for _ in range(W):
        orc.cpu_path(pos, off, idx, B, threads, per_step, False, use_ref)
    t0 = time.perf_counter()
    total = 0
    for _ in range(K):
        orc.cpu_path(pos, off, idx, B, threads, per_step, False, use_ref)
        total += threads * per_step * B
    dt = time.perf_counter() - t0
    value = total / dt
    rand = "reference random.cc compiled in place" if use_ref else "port"
    sample = (f"each step = {threads} threads x {per_step} batches of {B} (a bounded sample of the step's "
              f"{args.batches_per_step} batches) through pack (port) + Random executor ({rand}) + decode (port); no NN forward "
              "on the CPU: the reference has none, its CPU-runnable executor (Random, BASELINE.json configs[0]) stands in")
    line = {"impl": "reference", "metric": metric_name(B), "value": round(value, 1), "unit": UNIT, "n_gpus": args.gpus,
            "steps": K, "warmup": W, "ms_per_step": round(dt / K * 1e3, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args),
            "cpu_baseline": {"value": round(value, 1), "unit": UNIT, "cores": threads, "kind": "port",
                             "kind_detail": f"Random executor: {rand}; stage-1 pack and decode: ports (libnshogi absent)",
                             "sample": sample},
            "e2e": {"value": round(value, 1), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--batch", type=int, default=None)
    ap.add_argument("--channels", type=int, default=None)
    ap.add_argument("--blocks", type=int, default=None)
    ap.add_argument("--batches-per-step", type=int, default=None)
    ap.add_argument("--seed", type=int, default=None)
    ap.add_argument("--slots", type=int, default=4)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-selfplay", action="store_true")
    ap.add_argument("--no-latency-leg", action="store_true")
    ap.add_argument("--no-sweep", action="store_true")
    ap.add_argument("--selfplay-seconds", type=float, default=6.0)
    ap.add_argument("--small-pool", action="store_true", help="8-batch input pool (profiling runs only)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step's final batches (at most 8 and 64 MiB) to DIR/<name>.npy, float32: "
                         "legal_probs [batches, legal moves], win, draw, nan_flag [batches, batch]; the inputs depend on "
                         "the arguments only, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    c = CONFIGS[args.config]
    for k_arg, k_cfg in (("batch", "batch"), ("channels", "channels"), ("blocks", "blocks"), ("batches_per_step", "batches_per_step"),
                         ("seed", "seed")):
        if getattr(args, k_arg) is None:
            setattr(args, k_arg, c[k_cfg])
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
